// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[M,N] = op(A)[M,K] * op(B)[N,K]^T  (+bias) (*rowmask) (+residual)
//
// This is the dense-contraction workhorse behind every Linear of the ScorePerformer step
// (reference call sites: modules/transformer/attention.py:135-137,214; feedforward.py:19-21,56-61;
//  models/scoreperformer/embeddings.py:134-143,253-255,345-353; modules/layers.py:41-47).
//
// Layout per CTA (192 threads, 2 CTAs/SM):
//   warp 0      TMA producer   : cp.async.bulk.tensor 2D tiles, 128B swizzle, 3-stage mbarrier ring
//   warp 1      MMA issuer     : tcgen05.mma cta_group::1 kind::f16, M=128, N=BN, K=16; accumulator in TMEM
//   warps 2..5  epilogue       : tcgen05.ld 32x32b -> (bias) -> smem transpose -> (rowmask, residual) ->
//                                coalesced bf16/fp32 stores, or fp32 atomics for split-K
// Both operands may be K-major (row-major [rows, K]) or MN-major (row-major [K, rows]); the MN-major
// form feeds dgrad (B = W[out,in]) and wgrad (A = dY^T, B = X^T) without materialising transposes.
#include "common.cuh"

#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

namespace {

constexpr int BM = 128;
constexpr int BK = 64;       // 64 bf16 = 128 bytes = one SWIZZLE_128B atom row
constexpr int UMMA_K = 16;
constexpr int A_STAGE_BYTES = BM * BK * 2;
constexpr int EPI_WARPS = 8;                                  // two warps per TMEM lane quarter, one 64-column chunk each
constexpr int GEMM_THREADS = 64 + EPI_WARPS * 32;
constexpr int EPI_SST = 68;                                   // padded row stride (floats) of the direct epilogue's staging tile
// epilogue scratch: two 4 KB TMA boxes per warp + one row of bias per warp (TMA epilogue), which also covers the direct
// epilogue's one padded 32 x 64 fp32 chunk per warp
constexpr int EPI_BYTES = EPI_WARPS * 8192 + EPI_WARPS * 256 * 4;
static_assert(EPI_BYTES >= EPI_WARPS * 32 * EPI_SST * 4, "direct epilogue staging does not fit");

struct GemmParams {
    int M, N, K;
    int kb_per_split;      // k-blocks handled by one split
    int splits;
    void* C;
    int ldc;
    int c_fp32;            // 1: fp32 output, 0: bf16
    int atomic;            // 1: red.add fp32 (split-K / accumulate)
    const float* bias;     // [N] or null
    const float* residual; // fp32 [M, ldr] or null
    int ldr;
    const uint8_t* rowmask;  // [M] (bool) or null
    const float* alpha;      // device scalar multiplying the accumulator, or null
    float* rowdot_out;       // optional: out[(b*H + h)*T + t] = sum over the 64 columns of head h of C[m, :] * X[m, :] (m = b*T + t)
    int rd_T, rd_H;
    int tma_epi;             // 1: C (and the residual) go through TMA boxes; 0: direct vector stores
};

template <int BN>
__host__ __device__ constexpr int gemm_stages() {
    return BN == 256 ? 3 : (BN == 128 ? 4 : 6);
}
template <int BN>
constexpr int gemm_smem_bytes() {
    return gemm_stages<BN>() * (A_STAGE_BYTES + BN * BK * 2) + EPI_BYTES + 1024 /*align slack*/ + 512 /*barriers*/;
}

// Tile walk of one role: t = t0, t0 + step, ... decoded as (split, m-tile, n-tile) with n fastest.  The coordinates advance by
// carries instead of a division / modulo per tile (an integer division is ~40 instructions on the epilogue's critical path).
struct TileWalk {
    int split, m, n;
    int step_split, step_m, step_n, tiles_m, tiles_n;
    __device__ __forceinline__ TileWalk(int t0, int step, int tiles_m_, int tiles_n_) : tiles_m(tiles_m_), tiles_n(tiles_n_) {
        const int tiles_mn = tiles_m_ * tiles_n_;
        split = t0 / tiles_mn;
        int rem = t0 - split * tiles_mn;
        m = rem / tiles_n_;
        n = rem - m * tiles_n_;
        step_split = step / tiles_mn;
        rem = step - step_split * tiles_mn;
        step_m = rem / tiles_n_;
        step_n = rem - step_m * tiles_n_;
    }
    __device__ __forceinline__ void advance() {
        n += step_n;
        m += step_m;
        split += step_split;
        if (n >= tiles_n) { n -= tiles_n; ++m; }
        if (m >= tiles_m) { m -= tiles_m; ++split; }
    }
};

// Persistent, warp-specialised GEMM: one CTA per SM walks the tile list (n fastest, so co-running CTAs share the A panel in
// L2).  The TMA producer and the MMA issuer run ahead across tile boundaries; the accumulator is double-buffered in TMEM
// (2 x BN columns), so the epilogue of tile i overlaps the main loop of tile i+1.
template <int BN, bool A_MN, bool B_MN>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmR, GemmParams p) {
    constexpr int B_STAGE_BYTES = BN * BK * 2;
    constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
    constexpr int STAGES = gemm_stages<BN>();
    constexpr int TMEM_COLS = 2 * BN;            // double-buffered accumulator (BN = 256 uses all 512 columns)
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    float* epi_smem = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + EPI_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* acc_full = empty_bar + STAGES;     // [2]
    uint64_t* acc_empty = acc_full + 2;          // [2]
    uint64_t* res_bar = acc_empty + 2;           // [EPI_WARPS][2] residual boxes in flight
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(res_bar + 2 * EPI_WARPS);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int tiles_n = (p.N + BN - 1) / BN;
    const int tiles_m = (p.M + BM - 1) / BM;
    const int tiles_mn = tiles_m * tiles_n;
    const int total_tiles = tiles_mn * p.splits;
    const int total_kb = (p.K + BK - 1) / BK;
    const int tile0 = blockIdx.x, tile_step = gridDim.x;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&acc_full[a], 1);
            mbar_init(&acc_empty[a], EPI_WARPS);          // one arrive per epilogue warp
        }
        for (int a = 0; a < 2 * EPI_WARPS; ++a) mbar_init(&res_bar[a], 1);
        if (p.tma_epi) {
            tma_prefetch_desc(&tmC);
            if (p.residual != nullptr || p.rowdot_out != nullptr) tma_prefetch_desc(&tmR);
        }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<TMEM_COLS>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int s = 0;
            uint32_t phase = 0;
            TileWalk tw(tile0, tile_step, tiles_m, tiles_n);
            for (int t = tile0; t < total_tiles; t += tile_step, tw.advance()) {
                const int split = tw.split;
                const int m0 = tw.m * BM, n0 = tw.n * BN;
                const int kb0 = split * p.kb_per_split, kb1 = min(total_kb, kb0 + p.kb_per_split);
                for (int kb = kb0; kb < kb1; ++kb) {
                    mbar_wait(&empty_bar[s], phase ^ 1);
                    uint8_t* sA = smem + s * STAGE_BYTES;
                    uint8_t* sB = sA + A_STAGE_BYTES;
                    mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
                    if (A_MN) {
#pragma unroll
                        for (int h = 0; h < BM / 64; ++h) tma_load_2d(sA + h * (BK * 128), &tmA, &full_bar[s], m0 + h * 64, kb * BK);
                    } else {
                        tma_load_2d(sA, &tmA, &full_bar[s], kb * BK, m0);
                    }
                    if (B_MN) {
#pragma unroll
                        for (int h = 0; h < BN / 64; ++h) tma_load_2d(sB + h * (BK * 128), &tmB, &full_bar[s], n0 + h * 64, kb * BK);
                    } else {
                        tma_load_2d(sB, &tmB, &full_bar[s], kb * BK, n0);
                    }
                    if (++s == STAGES) { s = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, A_MN, B_MN);
            // K-major: 8-row groups are 1024 B apart (SBO); LBO unused.  MN-major: 64-element MN atoms
            // are BK*128 B apart (LBO), 8-k-row groups 1024 B apart (SBO).
            constexpr uint32_t a_lbo = A_MN ? BK * 128 : 0, b_lbo = B_MN ? BK * 128 : 0;
            constexpr uint32_t a_kstep = A_MN ? UMMA_K * 128 : UMMA_K * 2;   // bytes per UMMA_K step
            constexpr uint32_t b_kstep = B_MN ? UMMA_K * 128 : UMMA_K * 2;
            int s = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            TileWalk tw(tile0, tile_step, tiles_m, tiles_n);
            for (int t = tile0; t < total_tiles; t += tile_step, tw.advance()) {
                const int split = tw.split;
                const int kb0 = split * p.kb_per_split, kb1 = min(total_kb, kb0 + p.kb_per_split);
                mbar_wait(&acc_empty[acc], acc_phase ^ 1);       // epilogue has drained this accumulator buffer
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
                for (int i = 0; i < kb1 - kb0; ++i) {
                    mbar_wait(&full_bar[s], phase);
                    tc_fence_after();
                    const uint32_t a_addr = smem_u32(smem + s * STAGE_BYTES);
                    const uint32_t b_addr = a_addr + A_STAGE_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        const uint64_t da = umma_smem_desc_sw128(a_addr + k * a_kstep, a_lbo, 1024);
                        const uint64_t db = umma_smem_desc_sw128(b_addr + k * b_kstep, b_lbo, 1024);
                        umma_bf16(tmem_d, da, db, idesc, (i > 0 || k > 0) ? 1u : 0u);
                    }
                    umma_commit(&empty_bar[s]);
                    if (++s == STAGES) { s = 0; phase ^= 1; }
                }
                umma_commit(&acc_full[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ---------------- epilogue: warps 2..9; warp w may only touch TMEM lanes [32*(w%4), +32), i.e. thread = output row.
        // The two warps of a lane quarter alternate over the tile's column units.
        const int q = warp & 3;
        const int ew = warp - 2;
        const float alpha = p.alpha != nullptr ? __ldg(p.alpha) : 1.f;
        if (p.tma_epi) {
            // TMA epilogue.  Unit of work = one 4 KB box of C: 32 rows x 128 bytes (64 bf16 or 32 fp32 columns).  Each thread
            // converts its own row straight out of TMEM (+alpha, bias, rowmask, residual), writes it into a 128B-swizzled
            // staging box (conflict-free 16-byte stores) and one lane hands the box to the TMA unit: a plain tensor store, or
            // a tensor reduce-add for split-K / accumulate.  The residual tile arrives the same way (TMA load into the box
            // before it is overwritten), so every global access of the epilogue is a full-line asynchronous bulk transfer and
            // the warp is free to start the next unit while the previous box drains (two boxes per warp).
            constexpr int UNIT_STEP = EPI_WARPS / 4;
            constexpr int BIAS_PER_LANE = BN / 32;
            const int unit_first = ew >> 2;
            const int ucols = p.c_fp32 ? 32 : 64;
            const int units = BN / ucols;
            uint8_t* stage_w = reinterpret_cast<uint8_t*>(epi_smem) + ew * 8192;
            const uint32_t stage_a = smem_u32(stage_w);
            const uint32_t bias_a = smem_u32(reinterpret_cast<uint8_t*>(epi_smem) + EPI_WARPS * 8192) + (uint32_t)(ew * BN * 4);
            uint64_t* rbar = res_bar + ew * 2;
            const uint32_t sw = (uint32_t)(lane & 7);
            uint32_t rphase = 0;                 // bit b = parity of rbar[b]
            int ubuf = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            // the bias row of a tile is fetched one tile ahead (registers), so its global latency hides behind the previous tile
            float bias_next[BIAS_PER_LANE];
            auto fetch_bias = [&](int t, int n_tile) {
                const int n0 = n_tile * BN;
#pragma unroll
                for (int i = 0; i < BIAS_PER_LANE; ++i) {
                    const int c = n0 + i * 32 + lane;
                    bias_next[i] = (p.bias != nullptr && t < total_tiles && c < p.N) ? __ldg(p.bias + c) : 0.f;
                }
            };
            TileWalk tw(tile0, tile_step, tiles_m, tiles_n);
            fetch_bias(tile0, tw.n);
            for (int t = tile0; t < total_tiles; t += tile_step) {
                const int m0 = tw.m * BM, n0 = tw.n * BN;
                tw.advance();                        // tw now describes the NEXT tile of this CTA (bias prefetch below)
                const int row_base = m0 + q * 32;
                const int row = row_base + lane;
                if (p.bias != nullptr) {
#pragma unroll
                    for (int i = 0; i < BIAS_PER_LANE; ++i) sts_f1(bias_a + (uint32_t)((i * 32 + lane) * 4), bias_next[i]);
                }
                const bool keep = p.rowmask == nullptr || (row < p.M && p.rowmask[row] != 0);
                int last_u = -1;
                for (int u = unit_first; u < units && n0 + u * ucols < p.N; u += UNIT_STEP) last_u = u;
                __syncwarp();
                mbar_wait(&acc_full[acc], acc_phase);
                tc_fence_after();
                if (p.bias != nullptr) fetch_bias(t + tile_step, tw.n);
                const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(q * 32) << 16);
                if (last_u < 0 || row_base >= p.M) {
                    // nothing of this tile belongs to this warp: hand the accumulator back at once
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[acc]);
                    last_u = -1;
                }
#pragma unroll 1
                for (int u = unit_first; u <= last_u; u += UNIT_STEP) {
                    const int col0 = n0 + u * ucols;
                    uint8_t* st = stage_w + ubuf * 4096;
                    const uint32_t my = stage_a + (uint32_t)(ubuf * 4096 + lane * 128);
                    if (lane == 0) bulk_wait_group_read<1>();          // the store that last used this box has read it
                    __syncwarp();
                    if ((p.residual != nullptr || p.rowdot_out != nullptr) && lane == 0) {
                        // auxiliary input tile of this unit (fp32 residual, or the bf16 X of the fused row dot) -> the box
                        mbar_arrive_expect_tx(&rbar[ubuf], 4096);
                        tma_load_2d(st, &tmR, &rbar[ubuf], col0, row_base);
                    }
                    if (p.c_fp32) {
                        uint32_t v[32];
                        tmem_ld_32x32b_x32(tmem_acc + (uint32_t)(u * 32), v);
                        tmem_ld_wait();
                        if (u == last_u) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&acc_empty[acc]);
                        }
                        if (p.residual != nullptr) {
                            mbar_wait(&rbar[ubuf], (rphase >> ubuf) & 1u);
                            rphase ^= 1u << ubuf;
                        }
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                            if (p.bias != nullptr) b = lds_f4(bias_a + (uint32_t)((u * 32 + 4 * j) * 4));
                            float4 x;
                            x.x = fmaf(__uint_as_float(v[4 * j]), alpha, b.x);
                            x.y = fmaf(__uint_as_float(v[4 * j + 1]), alpha, b.y);
                            x.z = fmaf(__uint_as_float(v[4 * j + 2]), alpha, b.z);
                            x.w = fmaf(__uint_as_float(v[4 * j + 3]), alpha, b.w);
                            if (!keep) x = make_float4(0.f, 0.f, 0.f, 0.f);
                            const uint32_t slot = my + (((uint32_t)j ^ sw) << 4);
                            if (p.residual != nullptr) {
                                const float4 r = lds_f4(slot);
                                x.x += r.x; x.y += r.y; x.z += r.z; x.w += r.w;
                            }
                            sts_f4(slot, x);
                        }
                    } else {
                        uint32_t v[64];
                        tmem_ld_32x32b_x32(tmem_acc + (uint32_t)(u * 64), v);
                        tmem_ld_32x32b_x32(tmem_acc + (uint32_t)(u * 64 + 32), v + 32);
                        tmem_ld_wait();
                        if (u == last_u) {
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(&acc_empty[acc]);
                        }
                        if (p.rowdot_out != nullptr) {
                            mbar_wait(&rbar[ubuf], (rphase >> ubuf) & 1u);
                            rphase ^= 1u << ubuf;
                        }
                        float dot = 0.f;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
                            if (p.bias != nullptr) {
                                b0 = lds_f4(bias_a + (uint32_t)((u * 64 + 8 * j) * 4));
                                b1 = lds_f4(bias_a + (uint32_t)((u * 64 + 8 * j + 4) * 4));
                            }
                            float x[8];
                            x[0] = fmaf(__uint_as_float(v[8 * j]), alpha, b0.x); x[1] = fmaf(__uint_as_float(v[8 * j + 1]), alpha, b0.y);
                            x[2] = fmaf(__uint_as_float(v[8 * j + 2]), alpha, b0.z); x[3] = fmaf(__uint_as_float(v[8 * j + 3]), alpha, b0.w);
                            x[4] = fmaf(__uint_as_float(v[8 * j + 4]), alpha, b1.x); x[5] = fmaf(__uint_as_float(v[8 * j + 5]), alpha, b1.y);
                            x[6] = fmaf(__uint_as_float(v[8 * j + 6]), alpha, b1.z); x[7] = fmaf(__uint_as_float(v[8 * j + 7]), alpha, b1.w);
                            const uint32_t slot = my + (((uint32_t)j ^ sw) << 4);
                            if (p.rowdot_out != nullptr) {
                                // fused row dot (attention backward's delta = rowsum(dO * O)): X tile sits in the box we overwrite
                                const uint4 xr = lds_u4(slot);
                                const float2 a0 = unpack_bf16x2(xr.x), a1 = unpack_bf16x2(xr.y), a2 = unpack_bf16x2(xr.z), a3 = unpack_bf16x2(xr.w);
                                dot += x[0] * a0.x + x[1] * a0.y + x[2] * a1.x + x[3] * a1.y + x[4] * a2.x + x[5] * a2.y + x[6] * a3.x + x[7] * a3.y;
                            }
                            uint4 o;
                            o.x = pack_bf16x2(x[0], x[1]); o.y = pack_bf16x2(x[2], x[3]);
                            o.z = pack_bf16x2(x[4], x[5]); o.w = pack_bf16x2(x[6], x[7]);
                            if (!keep) o = make_uint4(0u, 0u, 0u, 0u);
                            sts_u4(slot, o);
                        }
                        if (p.rowdot_out != nullptr && row < p.M) {
                            const int bb = row / p.rd_T, tt = row - bb * p.rd_T;
                            p.rowdot_out[((size_t)bb * p.rd_H + (col0 >> 6)) * p.rd_T + tt] = keep ? dot : 0.f;
                        }
                    }
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) {
                        if (p.atomic) tma_reduce_add_2d(&tmC, st, col0, row_base);
                        else tma_store_2d(&tmC, st, col0, row_base);
                        bulk_commit_group();
                    }
                    ubuf ^= 1;
                }
                __syncwarp();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            if (lane == 0) bulk_wait_group<0>();
        } else {
            // Direct epilogue (fallback when C / residual do not meet the 16-byte TMA alignment rules): 64-column chunks go
            // TMEM -> registers -> padded smem (row stride 68 floats keeps float4 accesses conflict-free) -> 4 rows x 8 lanes
            // x 8 columns per pass, so a warp instruction covers four full 128/256-byte row segments.
            const int chunk_first = (warp - 2) >> 2;                 // 0 or 1
            constexpr int CHUNK_STEP = EPI_WARPS / 4;                // 2
            // Each warp drains its 32 accumulator rows 64 columns at a time: TMEM -> registers -> padded smem (row stride 68
            // floats keeps float4 accesses conflict-free) -> 4 rows x 8 lanes x 8 columns per pass, so every global access
            // is a 16/32-byte vector and a warp instruction covers four full 128/256-byte row segments.
            constexpr int SST = EPI_SST;
            float* stage = epi_smem + (warp - 2) * (32 * SST);
            float* Cf = reinterpret_cast<float*>(p.C);
            __nv_bfloat16* Cb = reinterpret_cast<__nv_bfloat16*>(p.C);
            const int sub_row = lane >> 3;          // 0..3
            const int sub_col = (lane & 7) * 8;     // 0..56
            const bool vec_ok = (p.ldc % 8 == 0) && (p.residual == nullptr || p.ldr % 4 == 0);
            int acc = 0;
            uint32_t acc_phase = 0;
            for (int t = tile0; t < total_tiles; t += tile_step) {
                const int rem = t % tiles_mn;      // (fallback path: keeps the plain decode)
                const int m0 = (rem / tiles_n) * BM, n0 = (rem % tiles_n) * BN;
                const int row_base = m0 + q * 32;
                mbar_wait(&acc_full[acc], acc_phase);
                tc_fence_after();
                const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * BN) + ((uint32_t)(q * 32) << 16);
                bool released = false;
    #pragma unroll 1
                for (int c = chunk_first; c < BN / 64 || !released; c += CHUNK_STEP) {
                    const int col0 = n0 + c * 64;
                    const bool live = c < BN / 64 && col0 < p.N;
                    if (live) {
                        uint32_t v[32];
    #pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            tmem_ld_32x32b_x32(tmem_acc + (uint32_t)(c * 64 + half * 32), v);
                            tmem_ld_wait();
    #pragma unroll
                            for (int j = 0; j < 32; j += 4)
                                *reinterpret_cast<float4*>(stage + lane * SST + half * 32 + j) =
                                    make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
                        }
                    }
                    if (!released && (c + CHUNK_STEP >= BN / 64 || n0 + (c + CHUNK_STEP) * 64 >= p.N)) {
                        // every accumulator value this warp needs is out of TMEM: hand the buffer back to the MMA warp
                        released = true;
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&acc_empty[acc]);
                    }
                    if (!live) break;
                    __syncwarp();
                    const int col = col0 + sub_col;
                    float bias[8];
    #pragma unroll
                    for (int j = 0; j < 8; ++j) bias[j] = (p.bias != nullptr && col + j < p.N) ? __ldg(p.bias + col + j) : 0.f;
                    const bool full = vec_ok && (col + 8 <= p.N);
    #pragma unroll 2
                    for (int it = 0; it < 8; ++it) {
                        const int r = it * 4 + sub_row;
                        const int row = row_base + r;
                        if (row >= p.M || col >= p.N) continue;
                        const float4 a0 = *reinterpret_cast<const float4*>(stage + r * SST + sub_col);
                        const float4 a1 = *reinterpret_cast<const float4*>(stage + r * SST + sub_col + 4);
                        float val[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                        const bool keep = p.rowmask == nullptr || p.rowmask[row] != 0;
    #pragma unroll
                        for (int j = 0; j < 8; ++j) val[j] = keep ? val[j] * alpha + bias[j] : 0.f;
                        const size_t off = (size_t)row * p.ldc + col;
                        if (full) {
                            if (p.residual != nullptr) {
                                const float4 r0 = *reinterpret_cast<const float4*>(p.residual + (size_t)row * p.ldr + col);
                                const float4 r1 = *reinterpret_cast<const float4*>(p.residual + (size_t)row * p.ldr + col + 4);
                                val[0] += r0.x; val[1] += r0.y; val[2] += r0.z; val[3] += r0.w;
                                val[4] += r1.x; val[5] += r1.y; val[6] += r1.z; val[7] += r1.w;
                            }
                            if (p.atomic) {   // split-K / accumulate: two 16-byte vector reductions per lane
                                asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(Cf + off), "f"(val[0]), "f"(val[1]), "f"(val[2]), "f"(val[3]) : "memory");
                                asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(Cf + off + 4), "f"(val[4]), "f"(val[5]), "f"(val[6]), "f"(val[7]) : "memory");
                            } else if (p.c_fp32) {
                                *reinterpret_cast<float4*>(Cf + off) = make_float4(val[0], val[1], val[2], val[3]);
                                *reinterpret_cast<float4*>(Cf + off + 4) = make_float4(val[4], val[5], val[6], val[7]);
                            } else {
                                uint4 o;
                                o.x = pack_bf16x2(val[0], val[1]); o.y = pack_bf16x2(val[2], val[3]);
                                o.z = pack_bf16x2(val[4], val[5]); o.w = pack_bf16x2(val[6], val[7]);
                                *reinterpret_cast<uint4*>(Cb + off) = o;
                            }
                        } else {
    #pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                if (col + j < p.N) {
                                    float vj = val[j];
                                    if (p.residual != nullptr) vj += p.residual[(size_t)row * p.ldr + col + j];
                                    if (p.atomic) atomicAdd(Cf + off + j, vj);
                                    else if (p.c_fp32) Cf[off + j] = vj;
                                    else Cb[off + j] = __float2bfloat16_rn(vj);
                                }
                            }
                        }
                    }
                    __syncwarp();
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }

        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<TMEM_COLS>(tmem_base);
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn == nullptr) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

template <int BN, bool A_MN, bool B_MN>
int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const CUtensorMap& tmR, const GemmParams& p,
                int splits, cudaStream_t stream) {
    auto kern = gemm_bf16_kernel<BN, A_MN, B_MN>;
    static bool configured = false;
    if (!configured) {
        SPB_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm_smem_bytes<BN>()));
        configured = true;
    }
    const int total_tiles = ceil_div(p.N, BN) * ceil_div(p.M, BM) * splits;
    const int grid = total_tiles < spb_num_sms() ? total_tiles : spb_num_sms();      // one CTA per SM
    kern<<<grid, GEMM_THREADS, gemm_smem_bytes<BN>(), stream>>>(tmA, tmB, tmC, tmR, p);
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}

}  // namespace

static int make_tmap_2d(CUtensorMap* out, CUtensorMapDataType dtype, const void* base, uint64_t inner, uint64_t outer,
                        uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer) {
    PFN_encodeTiled fn = get_encode_fn();
    if (fn == nullptr) {
        spb_set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)");
        return SPB_ERR_DRIVER;
    }
    SPB_CHECK_ARG((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA base pointer %p is not 16-byte aligned", base);
    SPB_CHECK_ARG((row_stride_bytes & 15) == 0, "TMA row stride %llu B is not a multiple of 16",
                  (unsigned long long)row_stride_bytes);
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {row_stride_bytes};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(out, dtype, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        spb_set_error("cuTensorMapEncodeTiled failed with CUresult %d (inner=%llu outer=%llu stride=%llu box=%ux%u)", (int)r,
                      (unsigned long long)inner, (unsigned long long)outer, (unsigned long long)row_stride_bytes, box_inner,
                      box_outer);
        return SPB_ERR_DRIVER;
    }
    return SPB_OK;
}

int spb_make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                          uint32_t box_inner, uint32_t box_outer) {
    return make_tmap_2d(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, inner, outer, row_stride_bytes, box_inner, box_outer);
}
int spb_make_tmap_f32_2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
                         uint32_t box_inner, uint32_t box_outer) {
    return make_tmap_2d(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, base, inner, outer, row_stride_bytes, box_inner, box_outer);
}

static int make_tmap_3d(CUtensorMap* out, CUtensorMapDataType dtype, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                        uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box0, uint32_t box1) {
    PFN_encodeTiled fn = get_encode_fn();
    if (fn == nullptr) {
        spb_set_error("cuTensorMapEncodeTiled is unavailable (driver too old?)");
        return SPB_ERR_DRIVER;
    }
    SPB_CHECK_ARG((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (stride1_bytes & 15) == 0 && (stride2_bytes & 15) == 0,
                  "TMA 3-D map: base / strides must be 16-byte aligned");
    cuuint64_t dims[3] = {d0, d1, d2};
    cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {box0, box1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(out, dtype, 3, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        spb_set_error("cuTensorMapEncodeTiled (3-D) failed with CUresult %d", (int)r);
        return SPB_ERR_DRIVER;
    }
    return SPB_OK;
}

int spb_make_tmap_bf16_3d(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                          uint64_t stride2_bytes, uint32_t box0, uint32_t box1) {
    return make_tmap_3d(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, d0, d1, d2, stride1_bytes, stride2_bytes, box0, box1);
}
int spb_make_tmap_f32_3d(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_bytes,
                         uint64_t stride2_bytes, uint32_t box0, uint32_t box1) {
    return make_tmap_3d(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, base, d0, d1, d2, stride1_bytes, stride2_bytes, box0, box1);
}

static int gemm_impl(const void* A, const void* B, void* C, int M, int N, int K, int trans_a, int trans_b, int lda, int ldb, int ldc,
                     const float* bias, const float* residual, int ldr, const uint8_t* rowmask, int c_fp32, int split_k, int accumulate,
                     const float* alpha, const void* rowdot_x, int ld_x, float* rowdot_out, int rd_T, int rd_H, cudaStream_t stream) {
    SPB_CHECK_ARG(A && B && C, "spb_gemm_bf16: null operand");
    SPB_CHECK_ARG(M > 0 && N > 0 && K > 0, "spb_gemm_bf16: empty problem M=%d N=%d K=%d", M, N, K);
    SPB_CHECK_ARG(lda % 8 == 0 && ldb % 8 == 0, "spb_gemm_bf16: lda=%d / ldb=%d must be multiples of 8 (TMA 16 B rule)", lda,
                  ldb);
    SPB_CHECK_ARG(!(accumulate || split_k > 1) || c_fp32, "spb_gemm_bf16: split-K / accumulate need an fp32 C");

    int BN = (N <= 64) ? 64 : 128;
    // wide tiles cut the L2->SM operand traffic per output.  SPB_GEMM_BN / SPB_GEMM_EPI override the heuristics for experiments.
    if (N % 256 == 0 && M >= 8 * BM) BN = 256;
    if (const char* e = getenv("SPB_GEMM_BN")) { int v = atoi(e); if (v == 64 || v == 128 || v == 256) BN = v; }
    const int total_kb = ceil_div(K, BK);
    int splits = 1;
    if (split_k > 1) splits = split_k;
    else if (split_k == 0 && c_fp32 && bias == nullptr && residual == nullptr && rowmask == nullptr) {
        // auto split-K for tall-K / small-output problems (wgrad)
        // one work item per SM measured best (fewer partial tiles to reduce-add into the same lines)
        const int tiles = ceil_div(M, BM) * ceil_div(N, BN), units = spb_num_sms();
        if (tiles < units && total_kb >= 8) splits = max(1, min(total_kb / 4, units / tiles));
    }
    int kb_per_split = ceil_div(total_kb, splits);
    splits = ceil_div(total_kb, kb_per_split);

    CUtensorMap tmA, tmB;
    int rc;
    if (trans_a) rc = spb_make_tmap_bf16_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)lda * 2, 64, BK);
    else rc = spb_make_tmap_bf16_2d(&tmA, A, (uint64_t)K, (uint64_t)M, (uint64_t)lda * 2, BK, BM);
    if (rc != SPB_OK) return rc;
    if (trans_b) rc = spb_make_tmap_bf16_2d(&tmB, B, (uint64_t)N, (uint64_t)K, (uint64_t)ldb * 2, 64, BK);
    else rc = spb_make_tmap_bf16_2d(&tmB, B, (uint64_t)K, (uint64_t)N, (uint64_t)ldb * 2, BK, (uint32_t)BN);
    if (rc != SPB_OK) return rc;

    // TMA epilogue whenever C (and the residual) satisfy the 16-byte base / row-pitch rules of a tensor map
    const size_t esize = c_fp32 ? 4 : 2;
    int tma_epi = ((reinterpret_cast<uintptr_t>(C) & 15) == 0 && ((size_t)ldc * esize) % 16 == 0) ? 1 : 0;
    if (residual != nullptr && !(c_fp32 && (reinterpret_cast<uintptr_t>(residual) & 15) == 0 && ((size_t)ldr * 4) % 16 == 0)) tma_epi = 0;
    if (const char* e = getenv("SPB_GEMM_EPI")) { if (e[0] == 'd') tma_epi = 0; }
    if (rowdot_out != nullptr) {
        SPB_CHECK_ARG(rowdot_x != nullptr && !c_fp32 && residual == nullptr && split_k <= 1 && !accumulate,
                      "spb_gemm_bf16_rowdot: needs a bf16 C without residual / split-K");
        SPB_CHECK_ARG(rd_T > 0 && rd_H > 0 && N == rd_H * 64 && M % rd_T == 0, "spb_gemm_bf16_rowdot: N must be H*64 and M a multiple of T");
        SPB_CHECK_ARG((reinterpret_cast<uintptr_t>(rowdot_x) & 15) == 0 && ld_x % 8 == 0, "spb_gemm_bf16_rowdot: X must be 16-byte aligned");
        SPB_CHECK_ARG(tma_epi, "spb_gemm_bf16_rowdot: C must satisfy the TMA alignment rules (16-byte base and row pitch)");
    }
    CUtensorMap tmC, tmR;
    memset(&tmC, 0, sizeof(tmC));
    memset(&tmR, 0, sizeof(tmR));
    if (tma_epi) {
        if (c_fp32) rc = spb_make_tmap_f32_2d(&tmC, C, (uint64_t)N, (uint64_t)M, (uint64_t)ldc * 4, 32, 32);
        else rc = spb_make_tmap_bf16_2d(&tmC, C, (uint64_t)N, (uint64_t)M, (uint64_t)ldc * 2, 64, 32);
        if (rc != SPB_OK) return rc;
        if (residual != nullptr) {
            rc = spb_make_tmap_f32_2d(&tmR, residual, (uint64_t)N, (uint64_t)M, (uint64_t)ldr * 4, 32, 32);
            if (rc != SPB_OK) return rc;
        } else if (rowdot_out != nullptr) {
            rc = spb_make_tmap_bf16_2d(&tmR, rowdot_x, (uint64_t)N, (uint64_t)M, (uint64_t)ld_x * 2, 64, 32);
            if (rc != SPB_OK) return rc;
        }
    }

    GemmParams p;
    p.M = M; p.N = N; p.K = K;
    p.kb_per_split = kb_per_split;
    p.splits = splits;
    p.C = C; p.ldc = ldc; p.c_fp32 = c_fp32;
    p.atomic = (splits > 1 || accumulate) ? 1 : 0;
    p.tma_epi = tma_epi;
    p.rowdot_out = rowdot_out; p.rd_T = rd_T; p.rd_H = rd_H;
    p.bias = bias; p.residual = residual; p.ldr = ldr; p.rowmask = rowmask; p.alpha = alpha;

    if (splits > 1 && !accumulate) {
        if (ldc == N) SPB_CHECK_CUDA(cudaMemsetAsync(C, 0, (size_t)M * N * sizeof(float), stream));
        else SPB_CHECK_CUDA(cudaMemset2DAsync(C, (size_t)ldc * 4, 0, (size_t)N * 4, M, stream));
    }

#define SPB_DISPATCH(BN_)                                                                                     \
    if (trans_a && trans_b) return launch_gemm<BN_, true, true>(tmA, tmB, tmC, tmR, p, splits, stream);      \
    if (trans_a) return launch_gemm<BN_, true, false>(tmA, tmB, tmC, tmR, p, splits, stream);                \
    if (trans_b) return launch_gemm<BN_, false, true>(tmA, tmB, tmC, tmR, p, splits, stream);                \
    return launch_gemm<BN_, false, false>(tmA, tmB, tmC, tmR, p, splits, stream);
    if (BN == 64) { SPB_DISPATCH(64) }
    if (BN == 256) { SPB_DISPATCH(256) }
    SPB_DISPATCH(128)
#undef SPB_DISPATCH
}

// C-ABI entry points; see include/spb200.h for the contracts.
extern "C" int spb_gemm_bf16(const void* A, const void* B, void* C, int M, int N, int K, int trans_a, int trans_b, int lda,
                             int ldb, int ldc, const float* bias, const float* residual, int ldr, const uint8_t* rowmask,
                             int c_fp32, int split_k, int accumulate, const float* alpha, cudaStream_t stream) {
    return gemm_impl(A, B, C, M, N, K, trans_a, trans_b, lda, ldb, ldc, bias, residual, ldr, rowmask, c_fp32, split_k, accumulate, alpha,
                     nullptr, 0, nullptr, 0, 0, stream);
}

// Same GEMM (bf16 C, no residual / split-K) whose epilogue also emits the per-head row dots
//   rowdot_out[(b*H + h)*T + t] = sum_{c in head h} C[b*T + t, c] * X[b*T + t, c]        (N == H*64)
// i.e. attention backward's delta = rowsum(dO * O) while dO = dY Wo is being produced (attend.py backward, flash form).
extern "C" int spb_gemm_bf16_rowdot(const void* A, const void* B, void* C, int M, int N, int K, int trans_a, int trans_b, int lda,
                                    int ldb, int ldc, const float* bias, const uint8_t* rowmask, const float* alpha, const void* X,
                                    int ld_x, float* rowdot_out, int T, int H, cudaStream_t stream) {
    SPB_CHECK_ARG(X && rowdot_out, "spb_gemm_bf16_rowdot: null X / rowdot_out");
    return gemm_impl(A, B, C, M, N, K, trans_a, trans_b, lda, ldb, ldc, bias, nullptr, 0, rowmask, 0, 1, 0, alpha, X, ld_x, rowdot_out, T,
                     H, stream);
}
