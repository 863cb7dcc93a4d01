// Fused feed-forward sub-layer for sm_100a (tcgen05 / TMEM / TMA):
//     out = resid + W2 . dropout( value * silu(gate) ),   [value | gate] = xn W1^T + b1
// Reference: modules/transformer/feedforward.py:13-22 (GLU), :35-64 (FeedForward: proj -> GLU -> dropout -> out) and the
// pre-norm residual around it, modules/transformer/transformer.py:139-232.
//
// A CTA pair (cluster of two, tcgen05 cta_group::2) owns 256 rows (note-tuples) at a time, 128 per CTA, and walks the tiles
// persistently.  The two weight matrices stream through shared memory in chunks of 64 hidden units; the [256 x 2048]
// pre-activation and the [256 x 1024] hidden activation never exist as a whole:
//   GEMM1(c)  u_c[256 x 128]   = xn[256 x 256] . W1_c^T      W1_c = value rows [64c, 64c+64) and gate rows [1024+64c, ..) stacked;
//                                                             xn stays resident in smem for the 16 chunks; accumulator in TMEM
//   GLU(c)    h_c[256 x 64]    = (u_val + b) * silu(u_gate + b) * keep      16 epilogue warps per CTA, one row per thread
//                                                             (TMEM lane == row), bf16 into a 128B-swizzled smem tile = the A
//                                                             operand of GEMM2
//   GEMM2(c)  acc[256 x 256]  += h_c[256 x 64] . W2[:, 64c:64c+64]^T         accumulates in TMEM over the 16 chunks
//   out       = acc + resid                                                   fp32, once per tile
// Each CTA stages its own 128 rows of xn / h and only HALF of every weight tile (CTA 0 the value rows of W1_c and output rows
// [0,128) of W2, CTA 1 the gate rows and output rows [128,256)), so the 1.5 MB of weights stream out of L2 once per 256 rows, and
// one tcgen05.mma issued by the leader CTA drives both SMs' tensor cores.  The leader issues GEMM1(c+1) before GEMM2(c), so the
// tensor pipe works on the next chunk while the epilogue warps run the GLU of this one (u is double-buffered in TMEM:
// 256 + 2 x 128 = 512 columns).
// For the backward (ffn_bwd.cu consumes u, the dW2 weight-gradient GEMM consumes h) the kernel can also emit u (bf16 [n, 2048],
// bias included) and h (bf16 [n, 1024]); both leave through TMA stores from staging tiles as whole 128-byte lines.
// HBM traffic per row: 512 B (xn) + 1 KB (resid) + 1 KB (out) [+ 4 KB u + 2 KB h when saved].
#include "attention_tc.cuh"
#include <string.h>

namespace {
using attn_tc::tmem_ld_32x32b_x16;

constexpr int D = 256;            // model width
constexpr int HID = 1024;         // hidden units (GLU: W1 has 2 * HID rows)
constexpr int BMF = 128;          // rows per CTA (a tile of the pair is 2 x BMF rows)
constexpr int CH = 64;            // hidden units per chunk
constexpr int NCH = HID / CH;     // 16 chunks
constexpr int KB1 = D / 64;       // 4 k-blocks of GEMM1
constexpr int EPQ = 4;            // epilogue warps per TMEM lane quarter
constexpr int FFN_EPI_WARPS = 4 * EPQ;
constexpr uint32_t TM_OUT = 0, TM_U = 256;

struct FfnParams {
    const float* bias1;          // [2 * HID]
    const float* resid;          // fp32 [n, ld_res] or null
    int ld_res;
    float* out;                  // fp32 [n, ld_out]
    int ld_out;
    __nv_bfloat16* u_save;       // bf16 [n, 2 * HID] or null
    __nv_bfloat16* h_save;       // bf16 [n, HID] or null
    int n_rows;
    uint64_t seed;
    const uint64_t* rng_offset;
    uint32_t thr32;              // drop when hash < thr32; 0 = dropout off
    float keep_scale;
};

constexpr int PW1_STAGES = 4;     // [64 rows x 64 k] 8 KB
constexpr int PW2_STAGES = 2;     // [128 rows x 64 k] 16 KB
constexpr int P_SA_OFF = 0;                                   // xn tile (own 128 rows)      64 KB
constexpr int P_SW1_OFF = P_SA_OFF + KB1 * 16384;             //                             48 KB
constexpr int P_SW2_OFF = P_SW1_OFF + PW1_STAGES * 8192;      //                             48 KB
constexpr int P_SH_OFF = P_SW2_OFF + PW2_STAGES * 16384;      // h chunks 2 x [128 x 64]     32 KB
constexpr int P_SU_OFF = P_SH_OFF + 2 * 16384;                // u staging: 2 x (value | gate)  64 KB
constexpr int P_SBIAS_OFF = P_SU_OFF + 4 * 16384;             //                              2 KB
constexpr int P_BAR_OFF = P_SBIAS_OFF + 2048;
constexpr int FFN_PAIR_SMEM_BYTES = P_BAR_OFF + 512;
static_assert(FFN_PAIR_SMEM_BYTES <= 232448, "exceeds the 227 KB of shared memory a CTA may have");
constexpr int FFN_PAIR_THREADS = 128 + FFN_EPI_WARPS * 32;    // producer, GEMM1 issuer, GEMM2 issuer, store thread, epilogue warps

__global__ void __launch_bounds__(FFN_PAIR_THREADS, 1)
ffn_fwd_pair_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW1, const __grid_constant__ CUtensorMap tmW2,
                    const __grid_constant__ CUtensorMap tmU, const __grid_constant__ CUtensorMap tmH, FfnParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + P_BAR_OFF);
    uint64_t* a_full = bars + 0;                       // leader
    uint64_t* a_empty = bars + 1;                      // both CTAs (multicast commit)
    uint64_t* w1_full = bars + 2;                      // [PW1_STAGES] leader
    uint64_t* w1_empty = w1_full + PW1_STAGES;         // both
    uint64_t* w2_full = w1_empty + PW1_STAGES;         // [PW2_STAGES] leader
    uint64_t* w2_empty = w2_full + PW2_STAGES;         // both
    uint64_t* u_full = w2_empty + PW2_STAGES;          // [2] both
    uint64_t* u_empty = u_full + 2;                    // [2] leader, one arrival per CTA (its forwarding thread)
    uint64_t* h_full = u_empty + 2;                    // [2] leader, one arrival per CTA
    uint64_t* h_empty = h_full + 2;                    // [2] both
    uint64_t* out_full = h_empty + 2;                  // both
    uint64_t* out_empty = out_full + 1;                // leader, 2 x 16 warps
    uint64_t* u_rd = out_empty + 1;                    // [2] local: u chunk read out by this CTA's 16 warps
    uint64_t* h_wr = u_rd + 2;                         // [2] local: h chunk (and the u staging tiles) written by this CTA's 16 warps
    uint64_t* st_empty = h_wr + 2;                     // [2] local: the chunk's TMA stores have read their tiles (staging b, h tile b)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(st_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int rank = (int)cluster_ctarank();
    const int n_ptiles = (p.n_rows + 2 * BMF - 1) / (2 * BMF);
    const int pt0 = blockIdx.x >> 1, pt_step = gridDim.x >> 1;
    const bool save = p.u_save != nullptr;

    if (threadIdx.x == 0) {
        if ((smem_u32(smem) & 1023u) != 0) {
            printf("spb200: ffn_fwd_pair_kernel needs 1024-byte aligned dynamic shared memory\n");
            __trap();
        }
        tma_prefetch_desc(&tmX);
        tma_prefetch_desc(&tmW1);
        tma_prefetch_desc(&tmW2);
        mbar_init(a_full, 1); mbar_init(a_empty, 1);
        for (int s = 0; s < PW1_STAGES; ++s) { mbar_init(&w1_full[s], 1); mbar_init(&w1_empty[s], 1); }
        for (int s = 0; s < PW2_STAGES; ++s) { mbar_init(&w2_full[s], 1); mbar_init(&w2_empty[s], 1); }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&u_full[b], 1); mbar_init(&u_empty[b], 2);
            mbar_init(&h_full[b], 2); mbar_init(&h_empty[b], 1);
            mbar_init(&u_rd[b], FFN_EPI_WARPS); mbar_init(&h_wr[b], FFN_EPI_WARPS);
        }
        mbar_init(out_full, 1); mbar_init(out_empty, 2 * FFN_EPI_WARPS);
        mbar_init(&st_empty[0], 1); mbar_init(&st_empty[1], 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc_pair<512>(tmem_slot);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer (both CTAs: own rows, own weight halves;
        // the byte counts land on the LEADER's full barriers, which gate the MMAs)
        if (lane == 0) {
            int s1 = 0, s2 = 0;
            uint32_t ph1 = 0, ph2 = 0;
            int it = 0;
            auto leader_bar = [](uint64_t* bar) { return smem_u32(bar) & 0xFEFFFFFFu; };     // same offset in the even CTA of the pair
            for (int pt = pt0; pt < n_ptiles; pt += pt_step, ++it) {
                const int m0 = pt * 2 * BMF + rank * BMF;
                auto load_w1 = [&](int c) {
                    for (int kb = 0; kb < KB1; ++kb) {
                        SPB_MBAR_WAIT(&w1_empty[s1], ph1 ^ 1u);
                        if (rank == 0) mbar_arrive_expect_tx(&w1_full[s1], 2 * 8192);
                        tma_load_2d_pair(smem + P_SW1_OFF + s1 * 8192, &tmW1, leader_bar(&w1_full[s1]), kb * 64, rank * HID + c * CH);
                        if (++s1 == PW1_STAGES) { s1 = 0; ph1 ^= 1u; }
                    }
                };
                load_w1(0);                                    // does not depend on the previous tile's xn being released
                SPB_MBAR_WAIT(a_empty, (uint32_t)(it & 1) ^ 1u);
                if (rank == 0) mbar_arrive_expect_tx(a_full, 2 * KB1 * 16384);
#pragma unroll
                for (int kb = 0; kb < KB1; ++kb) tma_load_2d_pair(smem + P_SA_OFF + kb * 16384, &tmX, leader_bar(a_full), kb * 64, m0);
                for (int c = 0; c < NCH; ++c) {
                    if (c > 0) load_w1(c);
                    SPB_MBAR_WAIT(&w2_empty[s2], ph2 ^ 1u);
                    if (rank == 0) mbar_arrive_expect_tx(&w2_full[s2], 2 * 16384);
                    tma_load_2d_pair(smem + P_SW2_OFF + s2 * 16384, &tmW2, leader_bar(&w2_full[s2]), c * CH, rank * BMF);
                    if (++s2 == PW2_STAGES) { s2 = 0; ph2 ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ GEMM1 issuer (leader CTA): u chunks for both CTAs
        if (lane == 0 && rank == 0) {
            constexpr uint32_t idesc1 = umma_idesc_bf16(2 * BMF, 2 * CH, false, false);
            const uint32_t sa = smem_u32(smem + P_SA_OFF), sw1 = smem_u32(smem + P_SW1_OFF);
            int s1 = 0;
            uint32_t ph1 = 0;
            int it = 0;
            for (int pt = pt0; pt < n_ptiles; pt += pt_step, ++it) {
                SPB_MBAR_WAIT(a_full, (uint32_t)(it & 1));
                for (int c = 0; c < NCH; ++c) {
                    const int g = it * NCH + c, b = g & 1;
                    SPB_MBAR_WAIT(&u_empty[b], (uint32_t)((g >> 1) & 1) ^ 1u);
                    tc_fence_after();
                    for (int kb = 0; kb < KB1; ++kb) {
                        SPB_MBAR_WAIT(&w1_full[s1], ph1);
                        tc_fence_after();
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            umma_bf16_pair(tmem_base + TM_U + b * 128, umma_smem_desc_sw128(sa + kb * 16384 + k * 32, 0, 1024),
                                           umma_smem_desc_sw128(sw1 + s1 * 8192 + k * 32, 0, 1024), idesc1, (kb > 0 || k > 0) ? 1u : 0u);
                        umma_commit_pair(&w1_empty[s1]);
                        if (++s1 == PW1_STAGES) { s1 = 0; ph1 ^= 1u; }
                    }
                    umma_commit_pair(&u_full[b]);
                }
                umma_commit_pair(a_empty);                 // every GEMM1 of this tile has been issued: xn may be replaced
            }
        }
    } else if (warp == 2) {
        // ------------------------------------------------------------------ GEMM2 issuer (leader CTA)
        if (lane == 0 && rank == 0) {
            constexpr uint32_t idesc2 = umma_idesc_bf16(2 * BMF, D, false, false);
            const uint32_t sw2 = smem_u32(smem + P_SW2_OFF), sh = smem_u32(smem + P_SH_OFF);
            int s2 = 0;
            uint32_t ph2 = 0;
            int it = 0;
            for (int pt = pt0; pt < n_ptiles; pt += pt_step, ++it) {
                for (int c = 0; c < NCH; ++c) {
                    const int g = it * NCH + c, b = g & 1;
                    SPB_MBAR_WAIT(&h_full[b], (uint32_t)((g >> 1) & 1));
                    SPB_MBAR_WAIT(&w2_full[s2], ph2);
                    if (c == 0) SPB_MBAR_WAIT(out_empty, (uint32_t)(it & 1) ^ 1u);
                    tc_fence_after();
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        umma_bf16_pair(tmem_base + TM_OUT, umma_smem_desc_sw128(sh + b * 16384 + k * 32, 0, 1024),
                                       umma_smem_desc_sw128(sw2 + s2 * 16384 + k * 32, 0, 1024), idesc2, (c > 0 || k > 0) ? 1u : 0u);
                    umma_commit_pair(&w2_empty[s2]);
                    umma_commit_pair(&h_empty[b]);
                    if (++s2 == PW2_STAGES) { s2 = 0; ph2 ^= 1u; }
                }
                umma_commit_pair(out_full);
            }
        }
    } else if (warp == 3) {
        // ------------------------------------------------------------------ forwarding / store thread (both CTAs).  The 16 epilogue
        // warps signal LOCAL barriers (a release at CTA scope is free); this thread turns each completed one into a single
        // cluster-scope arrival on the leader's barrier -- 16 cluster-scope release fences per chunk and CTA cost a third of the
        // kernel.  With side outputs it also sends the chunk's u / h tiles off through TMA.
        if (lane == 0) {
            if (save) {
                tma_prefetch_desc(&tmU);
                tma_prefetch_desc(&tmH);
            }
            const uint32_t u_empty_l[2] = {mapa_u32(&u_empty[0], 0), mapa_u32(&u_empty[1], 0)};
            const uint32_t h_full_l[2] = {mapa_u32(&h_full[0], 0), mapa_u32(&h_full[1], 0)};
            int it = 0;
            for (int pt = pt0; pt < n_ptiles; pt += pt_step, ++it) {
                const int m0 = pt * 2 * BMF + rank * BMF;
                for (int c = 0; c < NCH; ++c) {
                    const int g = it * NCH + c, b = g & 1;
                    const uint32_t ph = (uint32_t)((g >> 1) & 1);
                    SPB_MBAR_WAIT(&u_rd[b], ph);
                    mbar_arrive_cluster_relaxed(u_empty_l[b]);
                    SPB_MBAR_WAIT(&h_wr[b], ph);
                    mbar_arrive_cluster(h_full_l[b]);
                    if (save) {
                        if (m0 < p.n_rows) {
                            tma_store_2d(&tmU, smem + P_SU_OFF + b * 32768, c * CH, m0);
                            tma_store_2d(&tmU, smem + P_SU_OFF + b * 32768 + 16384, HID + c * CH, m0);
                            tma_store_2d(&tmH, smem + P_SH_OFF + b * 16384, c * CH, m0);
                            bulk_commit_group();
                            bulk_wait_group_read<0>();         // ~0.5 us: the tiles are handed back a whole chunk before they are needed
                        }
                        mbar_arrive(&st_empty[b]);
                    }
                }
            }
            if (save) bulk_wait_group<0>();
        }
    } else {
        // ------------------------------------------------------------------ epilogue warps (both CTAs, own 128 rows): thread == row
        constexpr int HW = CH / EPQ;                       // hidden units per warp and chunk
        constexpr int UW = EPQ == 2 ? 32 : 16;             // output columns per unit (4 units per warp)
        const int ew = warp - 4;
        const int q = warp & 3;                            // TMEM lane quarter this warp may touch
        const int part = ew >> 2;                          // which slice of the quarter's columns
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        const int r = q * 32 + lane;                       // row inside the CTA's tile
        float* sbias = reinterpret_cast<float*>(smem + P_SBIAS_OFF + ew * (2 * HW * 4));
        uint64_t seed = p.seed;
        if (p.rng_offset != nullptr) seed += *p.rng_offset * 0x9E3779B97F4A7C15ull;
        const uint32_t seed32 = spb_seed32(seed);
        const bool drop_on = p.thr32 != 0;
        const uint32_t sh_row = smem_u32(smem + P_SH_OFF) + (uint32_t)(r * 128);
        const uint32_t su_row = smem_u32(smem + P_SU_OFF) + (uint32_t)(r * 128);
        const uint32_t swz = (uint32_t)(r & 7);
        const uint32_t out_empty_l = mapa_u32(out_empty, 0);
        int it = 0;
        auto bias_at = [&](int c, int i) -> float {
            return i < 2 * HW ? __ldg(p.bias1 + (i < HW ? 0 : HID - HW) + c * CH + part * HW + i) : 0.f;
        };
        float bias_a = bias_at(0, lane), bias_b = bias_at(0, lane + 32);
        for (int pt = pt0; pt < n_ptiles; pt += pt_step, ++it) {
            const int row = pt * 2 * BMF + rank * BMF + r;
            const bool row_ok = row < p.n_rows;
            for (int c = 0; c < NCH; ++c) {
                const int g = it * NCH + c, b = g & 1;
                const uint32_t ph = (uint32_t)((g >> 1) & 1);
                const int hid0 = c * CH + part * HW;
                __syncwarp();
                if (lane < 2 * HW) sbias[lane] = bias_a;
                if (lane + 32 < 2 * HW) sbias[lane + 32] = bias_b;
                __syncwarp();
                {
                    const int cn = (c + 1 < NCH) ? c + 1 : 0;
                    bias_a = bias_at(cn, lane);
                    bias_b = bias_at(cn, lane + 32);
                }
                SPB_MBAR_WAIT(&u_full[b], ph);
                tc_fence_after();
                uint32_t val[HW], gat[HW];
                if (HW == 32) {
                    tmem_ld_32x32b_x32(tmem_base + TM_U + b * 128 + lane_addr + part * HW, val);
                    tmem_ld_32x32b_x32(tmem_base + TM_U + b * 128 + lane_addr + 64 + part * HW, gat);
                } else {
                    tmem_ld_32x32b_x16(tmem_base + TM_U + b * 128 + lane_addr + part * HW, val);
                    tmem_ld_32x32b_x16(tmem_base + TM_U + b * 128 + lane_addr + 64 + part * HW, gat);
                }
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&u_rd[b]);
                uint32_t hp[HW / 2];
                const uint32_t quad0 = (uint32_t)row * (uint32_t)(HID >> 2) + (uint32_t)(hid0 >> 2);
                const float4* sb4 = reinterpret_cast<const float4*>(sbias);
#pragma unroll
                for (int j = 0; j < HW; j += 4) {
                    const float4 bv = sb4[j >> 2], bg = sb4[(HW >> 2) + (j >> 2)];
                    const float bvs[4] = {bv.x, bv.y, bv.z, bv.w}, bgs[4] = {bg.x, bg.y, bg.z, bg.w};
                    float o[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float v = __uint_as_float(val[j + e]) + bvs[e];
                        const float gt = __uint_as_float(gat[j + e]) + bgs[e];
                        val[j + e] = __float_as_uint(v);
                        gat[j + e] = __float_as_uint(gt);
                        const float hg = 0.5f * gt;        // silu(g) = g/2 * (1 + tanh(g/2))
                        float th;
                        asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(hg));
                        o[e] = v * fmaf(hg, th, hg);
                    }
                    if (drop_on) {
                        const uint32_t qh = spb_quad_hash(seed32, quad0 + (uint32_t)(j >> 2));
#pragma unroll
                        for (int e = 0; e < 4; ++e) o[e] = spb_quad_keep(qh, e, p.thr32) ? o[e] * p.keep_scale : 0.f;
                    }
                    hp[j >> 1] = pack_bf16x2(o[0], o[1]);
                    hp[(j >> 1) + 1] = pack_bf16x2(o[2], o[3]);
                }
                SPB_MBAR_WAIT(&h_empty[b], ph ^ 1u);           // GEMM2 of the chunk that last used this h tile has completed
                if (save) SPB_MBAR_WAIT(&st_empty[b], ph ^ 1u);      // ... and the TMA stores of that chunk have read their tiles
#pragma unroll
                for (int j = 0; j < HW / 8; ++j) {
                    const uint32_t off = (((uint32_t)(part * (HW / 8) + j)) ^ swz) << 4;
                    sts_u4(sh_row + (uint32_t)(b * 16384) + off, make_uint4(hp[4 * j], hp[4 * j + 1], hp[4 * j + 2], hp[4 * j + 3]));
                    if (save) {
                        sts_u4(su_row + (uint32_t)(b * 32768) + off, make_uint4(pack_bf16x2(__uint_as_float(val[8 * j]), __uint_as_float(val[8 * j + 1])),
                                                        pack_bf16x2(__uint_as_float(val[8 * j + 2]), __uint_as_float(val[8 * j + 3])),
                                                        pack_bf16x2(__uint_as_float(val[8 * j + 4]), __uint_as_float(val[8 * j + 5])),
                                                        pack_bf16x2(__uint_as_float(val[8 * j + 6]), __uint_as_float(val[8 * j + 7]))));
                        sts_u4(su_row + (uint32_t)(b * 32768) + 16384 + off, make_uint4(pack_bf16x2(__uint_as_float(gat[8 * j]), __uint_as_float(gat[8 * j + 1])),
                                                                pack_bf16x2(__uint_as_float(gat[8 * j + 2]), __uint_as_float(gat[8 * j + 3])),
                                                                pack_bf16x2(__uint_as_float(gat[8 * j + 4]), __uint_as_float(gat[8 * j + 5])),
                                                                pack_bf16x2(__uint_as_float(gat[8 * j + 6]), __uint_as_float(gat[8 * j + 7]))));
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&h_wr[b]);
            }
            // ---- output: acc + resid -> fp32, this warp's 256 / EPQ columns of its 32 rows
            const bool use_res = p.resid != nullptr && row_ok;
            const float* rs = p.resid + (size_t)(row_ok ? row : 0) * p.ld_res + part * (D / EPQ);
            float* dst = p.out + (size_t)(row_ok ? row : 0) * p.ld_out + part * (D / EPQ);
            float4 rbuf[2][UW / 4];
            auto fetch_res = [&](int cu, float4 (&rb)[UW / 4]) {
#pragma unroll
                for (int j = 0; j < UW / 4; ++j)
                    rb[j] = use_res ? __ldg(reinterpret_cast<const float4*>(rs + cu * UW) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
            };
            fetch_res(0, rbuf[0]);
            SPB_MBAR_WAIT(out_full, (uint32_t)(it & 1));
            tc_fence_after();
#pragma unroll
            for (int cu = 0; cu < 4; ++cu) {
                if (cu + 1 < 4) fetch_res(cu + 1, rbuf[(cu + 1) & 1]);
                uint32_t v[UW];
                if (UW == 32) tmem_ld_32x32b_x32(tmem_base + TM_OUT + lane_addr + part * (D / EPQ) + cu * UW, v);
                else tmem_ld_32x32b_x16(tmem_base + TM_OUT + lane_addr + part * (D / EPQ) + cu * UW, v);
                tmem_ld_wait();
                if (cu == 3) {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive_cluster_relaxed(out_empty_l);
                }
                if (row_ok) {
#pragma unroll
                    for (int j = 0; j < UW / 4; ++j) {
                        const float4 rr = rbuf[cu & 1][j];
                        *reinterpret_cast<float4*>(dst + cu * UW + j * 4) =
                            make_float4(__uint_as_float(v[4 * j]) + rr.x, __uint_as_float(v[4 * j + 1]) + rr.y,
                                        __uint_as_float(v[4 * j + 2]) + rr.z, __uint_as_float(v[4 * j + 3]) + rr.w);
                    }
                }
            }
        }
    }
    __syncwarp();
    tc_fence_before();
    cluster_sync_all();              // the peer's smem / barriers must outlive the leader's last MMA and commit
    if (warp == 1) tmem_dealloc_pair<512>(tmem_base);
}

}  // namespace

// Fused feed-forward sub-layer forward (see the header of this file).  xn bf16 [n, 256] (ld_xn elements per row), w1 bf16
// [2048, 256] (value rows first, then gate rows: nn.Linear(dim, 2 * inner).weight of the GLU), b1 fp32 [2048], w2 bf16
// [256, 1024], resid fp32 [n, ld_res] or NULL, out fp32 [n, ld_out].  u_save (bf16 [n, 2048]) / h_save (bf16 [n, 1024]) may be
// NULL; when given they receive what the unfused path would have stored (pre-activation with bias; dropped hidden activation),
// with the same dropout mask function as spb_glu_fwd / spb_glu_bwd.
extern "C" int spb_ffn_fwd(const void* xn, int ld_xn, const void* w1, const float* b1, const void* w2, const float* resid, int ld_res,
                           float* out, int ld_out, void* u_save, void* h_save, int n_rows, int dim, int hidden, float dropout_p,
                           uint64_t seed, const uint64_t* rng_offset, cudaStream_t stream) {
    if (n_rows <= 0) return SPB_OK;
    SPB_CHECK_ARG(xn && w1 && b1 && w2 && out, "spb_ffn_fwd: null pointer");
    SPB_CHECK_ARG(dim == D && hidden == HID, "spb_ffn_fwd: built for dim 256 / hidden 1024 (got %d / %d)", dim, hidden);
    SPB_CHECK_ARG(ld_xn % 8 == 0 && ld_out % 4 == 0 && (resid == nullptr || ld_res % 4 == 0), "spb_ffn_fwd: bad leading dims");
    SPB_CHECK_ARG((reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(resid) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(u_save) & 15) == 0 && (reinterpret_cast<uintptr_t>(h_save) & 15) == 0,
                  "spb_ffn_fwd: out / resid / u_save / h_save must be 16-byte aligned");
    SPB_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, "spb_ffn_fwd: dropout_p must be in [0,1)");
    FfnParams p;
    p.bias1 = b1;
    p.resid = resid; p.ld_res = ld_res;
    p.out = out; p.ld_out = ld_out;
    p.u_save = reinterpret_cast<__nv_bfloat16*>(u_save);
    p.h_save = reinterpret_cast<__nv_bfloat16*>(h_save);
    p.n_rows = n_rows;
    p.seed = seed; p.rng_offset = rng_offset;
    p.thr32 = spb_drop_thr32(dropout_p);
    p.keep_scale = 1.f / (1.f - dropout_p);
    CUtensorMap tmX, tmW1, tmW2;
    int rc = spb_make_tmap_bf16_2d(&tmX, xn, (uint64_t)D, (uint64_t)n_rows, (uint64_t)ld_xn * 2, 64, BMF);
    if (rc != SPB_OK) return rc;
    rc = spb_make_tmap_bf16_2d(&tmW1, w1, (uint64_t)D, (uint64_t)(2 * HID), (uint64_t)D * 2, 64, CH);
    if (rc != SPB_OK) return rc;
    SPB_CHECK_ARG((u_save == nullptr) == (h_save == nullptr), "spb_ffn_fwd: u_save and h_save come together");
    rc = spb_make_tmap_bf16_2d(&tmW2, w2, (uint64_t)HID, (uint64_t)D, (uint64_t)HID * 2, 64, BMF);
    if (rc != SPB_OK) return rc;
    CUtensorMap tmU, tmH;
    memset(&tmU, 0, sizeof(tmU));
    memset(&tmH, 0, sizeof(tmH));
    if (u_save != nullptr) {
        rc = spb_make_tmap_bf16_2d(&tmU, u_save, (uint64_t)(2 * HID), (uint64_t)n_rows, (uint64_t)(2 * HID) * 2, 64, BMF);
        if (rc != SPB_OK) return rc;
        rc = spb_make_tmap_bf16_2d(&tmH, h_save, (uint64_t)HID, (uint64_t)n_rows, (uint64_t)HID * 2, 64, BMF);
        if (rc != SPB_OK) return rc;
    }
    SPB_CHECK_CUDA(cudaFuncSetAttribute(ffn_fwd_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FFN_PAIR_SMEM_BYTES));
    const int n_ptiles = ceil_div(n_rows, 2 * BMF);
    const int max_pairs = spb_num_sms() / 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * (n_ptiles < max_pairs ? n_ptiles : max_pairs));
    cfg.blockDim = dim3(FFN_PAIR_THREADS);
    cfg.dynamicSmemBytes = FFN_PAIR_SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SPB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, ffn_fwd_pair_kernel, tmX, tmW1, tmW2, tmU, tmH, p));
    SPB_CHECK_LAUNCH();
    return SPB_OK;
}
