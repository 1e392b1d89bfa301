// Fused multi-head attention backward for sm_100a (sequence length <= 1024, head dim 64 / 128 / 160).
//
// Flash-attention-2 style: with the log-sum-exp of every query row saved by the forward kernel and
// delta_i = sum_d dO_id * O_id, every [128 x 64] score tile can be rebuilt independently:
//     P = exp(S * hd^-1/2 - lse),   dS = P o (dP - delta) * hd^-1/2,   S = Q K^T,  dP = dO V^T.
// One kernel template, two roles (grid = (row blocks of 128, heads, images)):
//   kT = true  ("dK/dV"): a CTA owns 128 *keys*.   Resident X1 = K, X2 = V; streamed 64-query tiles Y1 = Q, Y2 = dO.
//                         T_s = K Q^T = S^T, T_p = V dO^T = dP^T;  dV += P^T dO,  dK += dS^T Q.
//   kT = false ("dQ")   : a CTA owns 128 *queries*. Resident X1 = Q, X2 = dO; streamed 64-key tiles Y1 = K, Y2 = V.
//                         T_s = Q K^T = S,   T_p = dO V^T = dP;    dQ += dS K.
// Both reductions therefore stay inside one CTA: no atomics, no cross-CTA exchange; the price is that S / dP are
// rebuilt by both roles (7 instead of 5 GEMM-equivalents -- tensor time is not what bounds these shapes).
//
// Pipeline (192 threads): warp 0 = TMA producer (resident tiles once, streamed tiles through a 2-stage ring),
// warp 1 = TMEM owner + tcgen05.mma issuer, warps 2-5 = one thread per resident row: tcgen05.ld of T_s / T_p,
// exp2 / dS math, bf16 P / dS staged in shared memory (K-major SWIZZLE_128B, one 64-column atom) as the A operand
// of the accumulating MMAs.  T_s is double-buffered in TMEM (except hd = 64, dK/dV role, where two CTAs per SM
// matter more), so the score MMA of tile j+1 runs under the exponentials of tile j.
// All operands are read in place from the packed qkv activation / the [tokens, D] gradient through 4-D tensor
// maps; streamed tiles serve both as K-major B (scores) and MN-major B (accumulation) without a transpose.
// Replaces: P re-materialisation + 4 batched GEMMs + softmax-backward kernel of the un-fused path
// (ops/cuda_ops.py:attention_bwd; reference: autograd through timm Attention, run_vit_training.py:134).
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>

#include "attention_sm100.h"
#include "gemm_sm100.h"
#include "ptx.cuh"

namespace b200 {

namespace {

constexpr int kBwdThreads = 192;
constexpr int kTileC = 64;    // streamed rows per tile == columns of a score tile
constexpr int kMaxSeq = 1024;  // column statistics of the dK/dV role live in shared memory: 2 * 4 B per token

struct AttnBwdParams {
    int N, H, B, D;
    float scale;       // hd^-1/2
    float scale_log2;  // hd^-1/2 * log2(e)
    const float* lse;    // [B*H, N] natural-log log-sum-exp of the scaled scores (forward kernel)
    const float* delta;  // [B*H, N] rowsum(dO o O)
    __nv_bfloat16* out1;  // kT: dK base (dqkv + D) / else dQ base (dqkv)
    __nv_bfloat16* out2;  // kT: dV base (dqkv + 2D)
    int64_t ld_out;       // 3 * D
};

template <int HD, bool kT>
struct BwdCfg {
    static constexpr int W = (HD % 64 == 0) ? 64 : 32;        // hd columns per swizzle atom
    static constexpr int kAtoms = HD / W;
    static constexpr uint32_t kLayout = (W == 64) ? 2u : 4u;
    static constexpr int kRowBytes = W * 2;
    static constexpr int kXBytes = 128 * HD * 2;              // one resident tile
    static constexpr int kYBytes = kTileC * HD * 2;           // one streamed tile
    static constexpr int kStageBytes = 2 * kYBytes;           // Y1 + Y2
    static constexpr int kEBytes = 128 * kTileC * 2;          // staged P / dS tile (16 KiB)
    static constexpr int kTsBufs = (kT && HD == 64) ? 1 : 2;
    static constexpr int kNumAcc = kT ? 2 : 1;
    static constexpr int kColTs = 0;
    static constexpr int kColTp = kTsBufs * kTileC;
    static constexpr int kColAcc1 = kColTp + kTileC;
    static constexpr int kColAcc2 = kColAcc1 + HD;
    static constexpr int kColsUsed = kColAcc1 + kNumAcc * HD;
    static constexpr int kTmemCols = kColsUsed <= 128 ? 128 : (kColsUsed <= 256 ? 256 : 512);
    // lse2 / delta of every query (column statistics of the dK/dV role), padded to whole tiles
    __host__ __device__ static constexpr int stat_bytes(int n_tokens) { return kT ? 2 * 4 * ((n_tokens + kTileC - 1) / kTileC) * kTileC : 0; }
    __host__ __device__ static constexpr int smem_bytes(int n_tokens) {
        return 2 * kXBytes + 2 * kStageBytes + 2 * kEBytes + stat_bytes(n_tokens) + 256;
    }
    static_assert(kColsUsed <= 512, "TMEM budget exceeded");
    static_assert(2 * kXBytes + 2 * kStageBytes + 2 * kEBytes + (kT ? 8 * kMaxSeq : 0) + 256 <= 232448,
                  "shared memory budget exceeded");
};

template <int HD, bool kT>
__global__ void __launch_bounds__(kBwdThreads) attn_bwd_sm100_kernel(const __grid_constant__ CUtensorMap tmap_x1,
                                                                    const __grid_constant__ CUtensorMap tmap_x2,
                                                                    const __grid_constant__ CUtensorMap tmap_y1,
                                                                    const __grid_constant__ CUtensorMap tmap_y2,
                                                                    const AttnBwdParams p) {
    using C = BwdCfg<HD, kT>;
    constexpr int W = C::W, kAtoms = C::kAtoms, kRowBytes = C::kRowBytes, kTsBufs = C::kTsBufs;
    constexpr uint32_t kLayout = C::kLayout;
    constexpr uint32_t kSbo = 8 * kRowBytes;

    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sX1 = smem;
    uint8_t* sX2 = sX1 + C::kXBytes;
    uint8_t* sY = sX2 + C::kXBytes;                 // [stage][Y1 | Y2]
    uint8_t* sE = sY + 2 * C::kStageBytes;          // P tile (A operand of the dV MMA; kT only)
    uint8_t* sD = sE + C::kEBytes;                  // dS tile (A operand of the dK / dQ MMA)
    const int nt = (p.N + kTileC - 1) / kTileC;
    float* s_lse2 = reinterpret_cast<float*>(sD + C::kEBytes);
    float* s_delta = s_lse2 + (kT ? nt * kTileC : 0);
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_lse2) + C::stat_bytes(p.N));
    uint64_t* bar_x = bars;            // resident tiles landed
    uint64_t* y_full = bars + 1;       // [2]
    uint64_t* y_empty = bars + 3;      // [2]
    uint64_t* ts_full = bars + 5;      // [2]
    uint64_t* ts_empty = bars + 7;     // [2]
    uint64_t* tp_full = bars + 9;
    uint64_t* tp_empty = bars + 10;
    uint64_t* e_full = bars + 11;
    uint64_t* e_empty = bars + 12;
    uint64_t* d_full = bars + 13;
    uint64_t* d_empty = bars + 14;
    uint64_t* acc_done = bars + 15;
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 16);

    const uint32_t warp_idx = threadIdx.x / 32;
    const uint32_t lane = lane_id();
    const int blk = blockIdx.x;  // which 128-row block of the resident operand
    const int h = blockIdx.y, b = blockIdx.z;
    const int64_t bh = static_cast<int64_t>(b) * p.H + h;

    if (warp_idx == 0 && elect_one()) {
        prefetch_tmap(&tmap_x1);
        prefetch_tmap(&tmap_x2);
        prefetch_tmap(&tmap_y1);
        prefetch_tmap(&tmap_y2);
        mbar_init(bar_x, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&y_full[i], 1);
            mbar_init(&y_empty[i], 1);
            mbar_init(&ts_full[i], 1);
            mbar_init(&ts_empty[i], 4);
        }
        mbar_init(tp_full, 1);
        mbar_init(tp_empty, 4);
        mbar_init(e_full, 4);
        mbar_init(e_empty, 1);
        mbar_init(d_full, 4);
        mbar_init(d_empty, 1);
        mbar_init(acc_done, 1);
        fence_mbar_init();
    }
    if (warp_idx == 1) tmem_alloc<1>(tmem_ptr_smem, C::kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp_idx == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            mbar_arrive_expect_tx(bar_x, 2 * C::kXBytes);
#pragma unroll
            for (int a = 0; a < kAtoms; ++a) {
                tma_load_4d(&tmap_x1, bar_x, sX1 + a * (128 * kRowBytes), a * W, blk * 128, h, b);
                tma_load_4d(&tmap_x2, bar_x, sX2 + a * (128 * kRowBytes), a * W, blk * 128, h, b);
            }
            for (int j = 0; j < nt; ++j) {
                const int st = j & 1;
                if (j >= 2) mbar_wait(&y_empty[st], ((j >> 1) - 1) & 1);
                uint8_t* y1 = sY + st * C::kStageBytes;
                uint8_t* y2 = y1 + C::kYBytes;
                mbar_arrive_expect_tx(&y_full[st], C::kStageBytes);
#pragma unroll
                for (int a = 0; a < kAtoms; ++a) {
                    tma_load_4d(&tmap_y1, &y_full[st], y1 + a * (kTileC * kRowBytes), a * W, j * kTileC, h, b);
                    tma_load_4d(&tmap_y2, &y_full[st], y2 + a * (kTileC * kRowBytes), a * W, j * kTileC, h, b);
                }
            }
        }
    } else if (warp_idx == 1) {
        // ===================================== MMA issuer =====================================
        if (elect_one()) {
            constexpr uint32_t idesc_t = make_idesc_bf16(128, kTileC, 0, 0);  // score tiles: both operands K-major
            constexpr uint32_t idesc_a = make_idesc_bf16(128, HD, 0, 1);      // accumulation: B = streamed tile, MN-major
            // T[128 x 64] = X[128 x hd] * Y[64 x hd]^T
            auto issue_scores = [&](uint32_t tmem_d, const uint8_t* sx, const uint8_t* sy) {
#pragma unroll
                for (int k = 0; k < HD / 16; ++k) {
                    const int atom = (k * 16) / W, within = (k * 16) % W;
                    const uint64_t da = make_smem_desc(smem_u32(sx) + atom * (128 * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    const uint64_t db = make_smem_desc(smem_u32(sy) + atom * (kTileC * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    umma_bf16<1>(tmem_d, da, db, idesc_t, k > 0 ? 1u : 0u);
                }
            };
            // acc[128 x hd] (+)= E[128 x 64] * Y[64 x hd]
            auto issue_acc = [&](uint32_t tmem_d, const uint8_t* se, const uint8_t* sy, bool accumulate) {
#pragma unroll
                for (int k = 0; k < kTileC / 16; ++k) {
                    const uint64_t da = make_smem_desc(smem_u32(se) + k * 32, 0, 1024, 2u);
                    // MN-major B: 8-row groups are 8*rowbytes apart (SBO), hd atoms are 64*rowbytes apart (LBO)
                    const uint64_t db = make_smem_desc(smem_u32(sy) + k * 16 * kRowBytes, kTileC * kRowBytes, kSbo, kLayout);
                    umma_bf16<1>(tmem_d, da, db, idesc_a, (accumulate || k > 0) ? 1u : 0u);
                }
            };
            mbar_wait(bar_x, 0);
            for (int j = 0; j < nt; ++j) {
                const int st = j & 1;
                const uint8_t* y1 = sY + st * C::kStageBytes;
                const uint8_t* y2 = y1 + C::kYBytes;
                if (j == 0) {
                    mbar_wait(&y_full[0], 0);
                    tc_fence_after();
                    issue_scores(tmem_base + C::kColTs, sX1, y1);
                    umma_commit<1>(&ts_full[0]);
                }
                if (j > 0) mbar_wait(tp_empty, (j - 1) & 1);
                tc_fence_after();
                issue_scores(tmem_base + C::kColTp, sX2, y2);
                umma_commit<1>(tp_full);
                if (j + 1 < nt) {  // score tile of the next streamed tile, under this tile's exponentials
                    const int j1 = j + 1, st1 = j1 & 1, tb1 = j1 % kTsBufs;
                    mbar_wait(&y_full[st1], (j1 >> 1) & 1);
                    if (j1 >= kTsBufs) mbar_wait(&ts_empty[tb1], (j1 / kTsBufs - 1) & 1);
                    tc_fence_after();
                    issue_scores(tmem_base + C::kColTs + tb1 * kTileC, sX1, sY + st1 * C::kStageBytes);
                    umma_commit<1>(&ts_full[tb1]);
                }
                if constexpr (kT) {
                    mbar_wait(e_full, j & 1);
                    tc_fence_after();
                    issue_acc(tmem_base + C::kColAcc2, sE, y2, j > 0);  // dV += P^T dO
                    umma_commit<1>(e_empty);
                }
                mbar_wait(d_full, j & 1);
                tc_fence_after();
                issue_acc(tmem_base + C::kColAcc1, sD, y1, j > 0);      // dK += dS^T Q   /   dQ += dS K
                umma_commit<1>(d_empty);
                umma_commit<1>(&y_empty[st]);
            }
            umma_commit<1>(acc_done);
        }
    } else {
        // ============================ softmax-backward math + epilogue ============================
        const uint32_t quarter = warp_idx & 3;
        const uint32_t r = quarter * 32 + lane;        // row of the resident block == TMEM lane
        const int row = blk * 128 + static_cast<int>(r);  // key index (kT) / query index
        const bool row_ok = row < p.N;
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16);
        constexpr float kLog2e = 1.4426950408889634f;
        float lse2_r = 0.f, delta_r = 0.f;
        if constexpr (kT) {
            // statistics are per *column* (query): stage all of them in shared memory once
            const int t = static_cast<int>(threadIdx.x) - 64;
            for (int q = t; q < nt * kTileC; q += 128) {
                const bool ok = q < p.N;
                s_lse2[q] = ok ? p.lse[bh * p.N + q] * kLog2e : 0.f;
                s_delta[q] = ok ? p.delta[bh * p.N + q] : 0.f;
            }
            named_bar_sync(1, 128);
        } else {
            if (row_ok) {
                lse2_r = p.lse[bh * p.N + row] * kLog2e;
                delta_r = p.delta[bh * p.N + row];
            }
        }
        const uint32_t erow = smem_u32(sE) + r * 128;
        const uint32_t drow = smem_u32(sD) + r * 128;
        for (int j = 0; j < nt; ++j) {
            const int tb = j % kTsBufs;
            uint32_t pk[kTileC / 2];  // bf16-rounded probabilities of this row, packed pairs
            mbar_wait(&ts_full[tb], (j / kTsBufs) & 1);
            tc_fence_after();
            if constexpr (kT) {
                if (j > 0) mbar_wait(e_empty, (j - 1) & 1);  // the dV MMA of the previous tile has consumed sE
            }
#pragma unroll
            for (int c = 0; c < kTileC / 32; ++c) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr + C::kColTs + tb * kTileC + c * 32, v);
                tmem_ld_wait();
#pragma unroll
                for (int i = 0; i < 32; i += 2) {
                    const int col = j * kTileC + c * 32 + i;  // streamed index: query (kT) / key
                    float l0, l1;
                    if constexpr (kT) {
                        l0 = s_lse2[col], l1 = s_lse2[col + 1];
                    } else {
                        l0 = l1 = lse2_r;
                    }
                    const float e0 = (row_ok && col < p.N) ? exp2f(fmaf(__uint_as_float(v[i]), p.scale_log2, -l0)) : 0.f;
                    const float e1 = (row_ok && col + 1 < p.N) ? exp2f(fmaf(__uint_as_float(v[i + 1]), p.scale_log2, -l1)) : 0.f;
                    pk[c * 16 + i / 2] = pack_bf16x2(e0, e1);
                }
                if constexpr (kT) {
#pragma unroll
                    for (int j8 = 0; j8 < 4; ++j8) {
                        const uint32_t chunk = c * 4 + j8;
                        st_shared_v4(erow + ((chunk ^ (r & 7)) << 4), pk[c * 16 + j8 * 4], pk[c * 16 + j8 * 4 + 1],
                                     pk[c * 16 + j8 * 4 + 2], pk[c * 16 + j8 * 4 + 3]);
                    }
                }
            }
            tc_fence_before();
            if constexpr (kT) fence_proxy_async_smem();  // generic-proxy writes -> tensor-core (async proxy) reads
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&ts_empty[tb]);
                if constexpr (kT) mbar_arrive(e_full);
            }

            mbar_wait(tp_full, j & 1);
            tc_fence_after();
            if (j > 0) mbar_wait(d_empty, (j - 1) & 1);
#pragma unroll
            for (int c = 0; c < kTileC / 32; ++c) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr + C::kColTp + c * 32, v);
                tmem_ld_wait();
                uint32_t dk[16];
#pragma unroll
                for (int i = 0; i < 32; i += 2) {
                    const int col = j * kTileC + c * 32 + i;
                    float d0, d1;
                    if constexpr (kT) {
                        d0 = s_delta[col], d1 = s_delta[col + 1];
                    } else {
                        d0 = d1 = delta_r;
                    }
                    const uint32_t pw = pk[c * 16 + i / 2];
                    // masked entries have P == 0, so dS == 0 there as well
                    const float s0 = bf16_lo(pw) * (__uint_as_float(v[i]) - d0) * p.scale;
                    const float s1 = bf16_hi(pw) * (__uint_as_float(v[i + 1]) - d1) * p.scale;
                    dk[i / 2] = pack_bf16x2(s0, s1);
                }
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    const uint32_t chunk = c * 4 + j8;
                    st_shared_v4(drow + ((chunk ^ (r & 7)) << 4), dk[j8 * 4], dk[j8 * 4 + 1], dk[j8 * 4 + 2],
                                 dk[j8 * 4 + 3]);
                }
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(tp_empty);
                mbar_arrive(d_full);
            }
        }

        // ---- epilogue: accumulators -> bf16 -> dqkv[token, head columns] ----
        mbar_wait(acc_done, 0);
        tc_fence_after();
#pragma unroll
        for (int a = 0; a < C::kNumAcc; ++a) {
            __nv_bfloat16* obase = (a == 0) ? p.out1 : p.out2;
            __nv_bfloat16* orow = obase + (static_cast<int64_t>(b) * p.N + row) * p.ld_out + h * HD;
            const uint32_t col0 = (a == 0) ? C::kColAcc1 : C::kColAcc2;
#pragma unroll 1
            for (int c = 0; c < HD / 32; ++c) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr + col0 + c * 32, v);
                tmem_ld_wait();
                if (row_ok) {
#pragma unroll
                    for (int j8 = 0; j8 < 4; ++j8) {
                        uint4 o;
                        o.x = pack_bf16x2(__uint_as_float(v[j8 * 8]), __uint_as_float(v[j8 * 8 + 1]));
                        o.y = pack_bf16x2(__uint_as_float(v[j8 * 8 + 2]), __uint_as_float(v[j8 * 8 + 3]));
                        o.z = pack_bf16x2(__uint_as_float(v[j8 * 8 + 4]), __uint_as_float(v[j8 * 8 + 5]));
                        o.w = pack_bf16x2(__uint_as_float(v[j8 * 8 + 6]), __uint_as_float(v[j8 * 8 + 7]));
                        *reinterpret_cast<uint4*>(orow + c * 32 + j8 * 8) = o;
                    }
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp_idx == 1) tmem_dealloc<1>(tmem_base, C::kTmemCols);
}

// ------------------------------------------------------------------------------------------------
// Long-sequence forward (N > 256, e.g. 576 tokens at 336 px): two passes over the 64-key tiles instead of an online
// softmax.  Pass 1 rebuilds S = Q K^T tile by tile and keeps only the running row max / sum (-> log-sum-exp);
// pass 2 rebuilds S again, writes P = exp(S - lse) (already normalised) as the A operand and accumulates O += P V in
// TMEM with no rescaling.  Same warp roles, TMA ring and TMEM double-buffering as the backward kernel above; scores
// never reach HBM (the un-fused path materialises a [B, H, N, N] tensor: 2.6 GiB per ViT-10B block at 336 px).
// ------------------------------------------------------------------------------------------------
struct AttnFwdLongParams {
    int N, H, B, D;
    float scale_log2;
    __nv_bfloat16* out;  // [B*N, D]
    float* lse;          // [B*H, N]
};

template <int HD>
struct FwdLongCfg {
    static constexpr int W = (HD % 64 == 0) ? 64 : 32;
    static constexpr int kAtoms = HD / W;
    static constexpr uint32_t kLayout = (W == 64) ? 2u : 4u;
    static constexpr int kRowBytes = W * 2;
    static constexpr int kXBytes = 128 * HD * 2;
    static constexpr int kYBytes = kTileC * HD * 2;
    static constexpr int kStageBytes = 2 * kYBytes;  // K tile + V tile
    static constexpr int kEBytes = 128 * kTileC * 2;
    static constexpr int kColAcc = 2 * kTileC;
    static constexpr int kTmemCols = (kColAcc + HD) <= 256 ? 256 : 512;
    static constexpr int kSmem = kXBytes + 2 * kStageBytes + kEBytes + 256;
    static_assert(kSmem <= 232448, "shared memory budget exceeded");
};

template <int HD>
__global__ void __launch_bounds__(kBwdThreads) attn_fwd_long_sm100_kernel(const __grid_constant__ CUtensorMap tmap_q,
                                                                         const __grid_constant__ CUtensorMap tmap_k,
                                                                         const __grid_constant__ CUtensorMap tmap_v,
                                                                         const AttnFwdLongParams p) {
    using C = FwdLongCfg<HD>;
    constexpr int W = C::W, kAtoms = C::kAtoms, kRowBytes = C::kRowBytes;
    constexpr uint32_t kLayout = C::kLayout;
    constexpr uint32_t kSbo = 8 * kRowBytes;

    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sQ = smem;
    uint8_t* sY = sQ + C::kXBytes;               // [stage][K | V]
    uint8_t* sE = sY + 2 * C::kStageBytes;       // P tile
    uint64_t* bars = reinterpret_cast<uint64_t*>(sE + C::kEBytes);
    uint64_t* bar_x = bars;
    uint64_t* y_full = bars + 1;    // [2]
    uint64_t* y_empty = bars + 3;   // [2]
    uint64_t* ts_full = bars + 5;   // [2]
    uint64_t* ts_empty = bars + 7;  // [2]
    uint64_t* e_full = bars + 9;
    uint64_t* e_empty = bars + 10;
    uint64_t* acc_done = bars + 11;
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 12);

    const uint32_t warp_idx = threadIdx.x / 32;
    const uint32_t lane = lane_id();
    const int blk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
    const int nt = (p.N + kTileC - 1) / kTileC;
    const int nl = 2 * nt;  // tile visits: pass 1 (K only), pass 2 (K and V)

    if (warp_idx == 0 && elect_one()) {
        prefetch_tmap(&tmap_q);
        prefetch_tmap(&tmap_k);
        prefetch_tmap(&tmap_v);
        mbar_init(bar_x, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&y_full[i], 1);
            mbar_init(&y_empty[i], 1);
            mbar_init(&ts_full[i], 1);
            mbar_init(&ts_empty[i], 4);
        }
        mbar_init(e_full, 4);
        mbar_init(e_empty, 1);
        mbar_init(acc_done, 1);
        fence_mbar_init();
    }
    if (warp_idx == 1) tmem_alloc<1>(tmem_ptr_smem, C::kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp_idx == 0) {
        if (elect_one()) {
            mbar_arrive_expect_tx(bar_x, C::kXBytes);
#pragma unroll
            for (int a = 0; a < kAtoms; ++a)
                tma_load_4d(&tmap_q, bar_x, sQ + a * (128 * kRowBytes), a * W, blk * 128, h, b);
            for (int l = 0; l < nl; ++l) {
                const int st = l & 1, tile = l % nt;
                const bool with_v = l >= nt;
                if (l >= 2) mbar_wait(&y_empty[st], ((l >> 1) - 1) & 1);
                uint8_t* yk = sY + st * C::kStageBytes;
                uint8_t* yv = yk + C::kYBytes;
                mbar_arrive_expect_tx(&y_full[st], with_v ? C::kStageBytes : C::kYBytes);
#pragma unroll
                for (int a = 0; a < kAtoms; ++a) {
                    tma_load_4d(&tmap_k, &y_full[st], yk + a * (kTileC * kRowBytes), a * W, tile * kTileC, h, b);
                    if (with_v)
                        tma_load_4d(&tmap_v, &y_full[st], yv + a * (kTileC * kRowBytes), a * W, tile * kTileC, h, b);
                }
            }
        }
    } else if (warp_idx == 1) {
        if (elect_one()) {
            constexpr uint32_t idesc_t = make_idesc_bf16(128, kTileC, 0, 0);
            constexpr uint32_t idesc_a = make_idesc_bf16(128, HD, 0, 1);
            auto issue_scores = [&](uint32_t tmem_d, const uint8_t* sy) {
#pragma unroll
                for (int k = 0; k < HD / 16; ++k) {
                    const int atom = (k * 16) / W, within = (k * 16) % W;
                    const uint64_t da = make_smem_desc(smem_u32(sQ) + atom * (128 * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    const uint64_t db = make_smem_desc(smem_u32(sy) + atom * (kTileC * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    umma_bf16<1>(tmem_d, da, db, idesc_t, k > 0 ? 1u : 0u);
                }
            };
            mbar_wait(bar_x, 0);
            for (int l = 0; l < nl; ++l) {
                const int st = l & 1;
                if (l == 0) {
                    mbar_wait(&y_full[0], 0);
                    tc_fence_after();
                    issue_scores(tmem_base, sY);
                    umma_commit<1>(&ts_full[0]);
                }
                if (l < nt) umma_commit<1>(&y_empty[st]);  // pass 1: the K tile is free once its score MMA is done
                if (l + 1 < nl) {
                    const int l1 = l + 1, s1 = l1 & 1;
                    mbar_wait(&y_full[s1], (l1 >> 1) & 1);
                    if (l1 >= 2) mbar_wait(&ts_empty[s1], ((l1 >> 1) - 1) & 1);
                    tc_fence_after();
                    issue_scores(tmem_base + s1 * kTileC, sY + s1 * C::kStageBytes);
                    umma_commit<1>(&ts_full[s1]);
                }
                if (l >= nt) {
                    const int i = l - nt;
                    const uint8_t* yv = sY + st * C::kStageBytes + C::kYBytes;
                    mbar_wait(e_full, i & 1);
                    tc_fence_after();
#pragma unroll
                    for (int k = 0; k < kTileC / 16; ++k) {
                        const uint64_t da = make_smem_desc(smem_u32(sE) + k * 32, 0, 1024, 2u);
                        const uint64_t db = make_smem_desc(smem_u32(yv) + k * 16 * kRowBytes, kTileC * kRowBytes, kSbo, kLayout);
                        umma_bf16<1>(tmem_base + C::kColAcc, da, db, idesc_a, (i > 0 || k > 0) ? 1u : 0u);
                    }
                    umma_commit<1>(e_empty);
                    umma_commit<1>(&y_empty[st]);
                }
            }
            umma_commit<1>(acc_done);
        }
    } else {
        const uint32_t quarter = warp_idx & 3;
        const uint32_t r = quarter * 32 + lane;
        const int q = blk * 128 + static_cast<int>(r);
        const bool row_ok = q < p.N;
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16);
        const uint32_t erow = smem_u32(sE) + r * 128;
        // ---- pass 1: running max / sum of the scaled scores (log2 domain) ----
        float mx = -INFINITY, sum = 0.f;
        for (int l = 0; l < nt; ++l) {
            mbar_wait(&ts_full[l & 1], (l >> 1) & 1);
            tc_fence_after();
            uint32_t v0[32], v1[32];
            tmem_ld_32x32b_x32(taddr + (l & 1) * kTileC, v0);
            tmem_ld_32x32b_x32(taddr + (l & 1) * kTileC + 32, v1);
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&ts_empty[l & 1]);  // values are in registers: the buffer may be overwritten
            float tmax = -INFINITY;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (l * kTileC + i < p.N) tmax = fmaxf(tmax, __uint_as_float(v0[i]));
                if (l * kTileC + 32 + i < p.N) tmax = fmaxf(tmax, __uint_as_float(v1[i]));
            }
            const float m_new = fmaxf(mx, tmax);
            const float ms = m_new * p.scale_log2;
            float part = 0.f;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (l * kTileC + i < p.N) part += exp2f(fmaf(__uint_as_float(v0[i]), p.scale_log2, -ms));
                if (l * kTileC + 32 + i < p.N) part += exp2f(fmaf(__uint_as_float(v1[i]), p.scale_log2, -ms));
            }
            sum = sum * exp2f((mx - m_new) * p.scale_log2) + part;  // first tile: mx = -inf -> factor 0
            mx = m_new;
        }
        const float lse2 = mx * p.scale_log2 + log2f(sum);
        // ---- pass 2: P = exp2(S * c - lse2) -> shared memory -> O += P V ----
        for (int l = nt; l < nl; ++l) {
            const int i = l - nt;
            mbar_wait(&ts_full[l & 1], (l >> 1) & 1);
            tc_fence_after();
            if (i > 0) mbar_wait(e_empty, (i - 1) & 1);
#pragma unroll
            for (int c = 0; c < kTileC / 32; ++c) {
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr + (l & 1) * kTileC + c * 32, v);
                tmem_ld_wait();
                uint32_t pk[16];
#pragma unroll
                for (int t = 0; t < 32; t += 2) {
                    const int col = i * kTileC + c * 32 + t;
                    const float e0 = col < p.N ? exp2f(fmaf(__uint_as_float(v[t]), p.scale_log2, -lse2)) : 0.f;
                    const float e1 = col + 1 < p.N ? exp2f(fmaf(__uint_as_float(v[t + 1]), p.scale_log2, -lse2)) : 0.f;
                    pk[t / 2] = pack_bf16x2(e0, e1);
                }
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    const uint32_t chunk = c * 4 + j8;
                    st_shared_v4(erow + ((chunk ^ (r & 7)) << 4), pk[j8 * 4], pk[j8 * 4 + 1], pk[j8 * 4 + 2],
                                 pk[j8 * 4 + 3]);
                }
            }
            tc_fence_before();
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&ts_empty[l & 1]);
                mbar_arrive(e_full);
            }
        }
        // ---- epilogue ----
        const int64_t bh = static_cast<int64_t>(b) * p.H + h;
        if (row_ok) p.lse[bh * p.N + q] = lse2 * 0.6931471805599453f;
        mbar_wait(acc_done, 0);
        tc_fence_after();
        __nv_bfloat16* orow = p.out + (static_cast<int64_t>(b) * p.N + q) * p.D + h * HD;
#pragma unroll 1
        for (int c = 0; c < HD / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32b_x32(taddr + C::kColAcc + c * 32, v);
            tmem_ld_wait();
            if (row_ok) {
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    uint4 o;
                    o.x = pack_bf16x2(__uint_as_float(v[j8 * 8]), __uint_as_float(v[j8 * 8 + 1]));
                    o.y = pack_bf16x2(__uint_as_float(v[j8 * 8 + 2]), __uint_as_float(v[j8 * 8 + 3]));
                    o.z = pack_bf16x2(__uint_as_float(v[j8 * 8 + 4]), __uint_as_float(v[j8 * 8 + 5]));
                    o.w = pack_bf16x2(__uint_as_float(v[j8 * 8 + 6]), __uint_as_float(v[j8 * 8 + 7]));
                    *reinterpret_cast<uint4*>(orow + c * 32 + j8 * 8) = o;
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp_idx == 1) tmem_dealloc<1>(tmem_base, C::kTmemCols);
}

// delta[bh, q] = sum_d dO[token, h*hd + d] * O[token, h*hd + d]; 4 lanes per (token, head)
__global__ void attn_delta_kernel(const __nv_bfloat16* __restrict__ dout, int64_t ld_do,
                                  const __nv_bfloat16* __restrict__ out, int64_t ld_o, float* __restrict__ delta,
                                  const float* __restrict__ lse, float* __restrict__ lse2, int B, int N, int H, int hd) {
    const int64_t gid = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) / 4;
    const int sub = threadIdx.x & 3;
    const int64_t total = static_cast<int64_t>(B) * N * H;
    float acc = 0.f;
    if (gid < total) {
        const int hh = static_cast<int>(gid % H);
        const int64_t token = gid / H;
        const uint4* a = reinterpret_cast<const uint4*>(dout + token * ld_do + hh * hd);
        const uint4* o = reinterpret_cast<const uint4*>(out + token * ld_o + hh * hd);
        for (int c = sub; c < hd / 8; c += 4) {
            const uint4 x = a[c], y = o[c];
            const uint32_t xs[4] = {x.x, x.y, x.z, x.w}, ys[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
            for (int t = 0; t < 4; ++t) acc += bf16_lo(xs[t]) * bf16_lo(ys[t]) + bf16_hi(xs[t]) * bf16_hi(ys[t]);
        }
    }
    acc += __shfl_xor_sync(0xffffffffu, acc, 1);
    acc += __shfl_xor_sync(0xffffffffu, acc, 2);
    if (gid < total && sub == 0) {
        const int hh = static_cast<int>(gid % H);
        const int64_t token = gid / H;
        const int64_t bb = token / N, q = token % N;
        delta[(bb * H + hh) * N + q] = acc;
        // the persistent backward wants the row log-sum-exp in log2 units, bulk-copyable: write it alongside
        if (lse2 != nullptr) lse2[(bb * H + hh) * N + q] = lse[(bb * H + hh) * N + q] * 1.4426950408889634f;
    }
}

template <int HD, bool kT>
void launch_bwd(const GemmOperand& x1, const GemmOperand& x2, const GemmOperand& y1, const GemmOperand& y2,
                const AttnBwdParams& p, cudaStream_t stream) {
    using C = BwdCfg<HD, kT>;
    auto kern = attn_bwd_sm100_kernel<HD, kT>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::smem_bytes(kMaxSeq));
        if (err != cudaSuccess)
            throw std::runtime_error(std::string("attention bwd smem attr: ") + cudaGetErrorString(err));
        attr_set = true;
    }
    const int sw = C::W * 2;
    CUtensorMap tx1 = make_tensor_map_4d(x1, HD, p.N, C::W, 128, sw);
    CUtensorMap tx2 = make_tensor_map_4d(x2, HD, p.N, C::W, 128, sw);
    CUtensorMap ty1 = make_tensor_map_4d(y1, HD, p.N, C::W, kTileC, sw);
    CUtensorMap ty2 = make_tensor_map_4d(y2, HD, p.N, C::W, kTileC, sw);
    dim3 grid((p.N + 127) / 128, p.H, p.B);
    kern<<<grid, kBwdThreads, C::smem_bytes(p.N), stream>>>(tx1, tx2, ty1, ty2, p);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) throw std::runtime_error(std::string("attention bwd launch: ") + cudaGetErrorString(err));
}

template <int HD>
void run_bwd(const GemmOperand& q, const GemmOperand& k, const GemmOperand& v, const GemmOperand& dO,
             AttnBwdParams p, __nv_bfloat16* dqkv, cudaStream_t stream) {
    p.out1 = dqkv + p.D, p.out2 = dqkv + 2 * p.D;
    launch_bwd<HD, true>(k, v, q, dO, p, stream);   // dK, dV
    p.out1 = dqkv, p.out2 = nullptr;
    launch_bwd<HD, false>(q, dO, k, v, p, stream);  // dQ
}

template <int HD>
void launch_fwd_long(const GemmOperand& q, const GemmOperand& k, const GemmOperand& v, const AttnFwdLongParams& p,
                     cudaStream_t stream) {
    using C = FwdLongCfg<HD>;
    auto kern = attn_fwd_long_sm100_kernel<HD>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmem);
        if (err != cudaSuccess)
            throw std::runtime_error(std::string("attention fwd-long smem attr: ") + cudaGetErrorString(err));
        attr_set = true;
    }
    const int sw = C::W * 2;
    CUtensorMap tq = make_tensor_map_4d(q, HD, p.N, C::W, 128, sw);
    CUtensorMap tk = make_tensor_map_4d(k, HD, p.N, C::W, kTileC, sw);
    CUtensorMap tv = make_tensor_map_4d(v, HD, p.N, C::W, kTileC, sw);
    dim3 grid((p.N + 127) / 128, p.H, p.B);
    kern<<<grid, kBwdThreads, C::kSmem, stream>>>(tq, tk, tv, p);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess)
        throw std::runtime_error(std::string("attention fwd-long launch: ") + cudaGetErrorString(err));
}

bool attention_fwd_long_supported(int N, int hd) { return N % 2 == 0 && (hd == 64 || hd == 128 || hd == 160); }

bool attention_bwd_supported(int N, int hd) {
    return N <= kMaxSeq && N % 2 == 0 && (hd == 64 || hd == 128 || hd == 160);
}

}  // namespace

void attention_fwd_long(const __nv_bfloat16* qkv, int64_t ld_qkv, __nv_bfloat16* out, float* lse, int B, int N, int H,
                        int hd, cudaStream_t stream) {
    if (!attention_fwd_long_supported(N, hd)) throw std::runtime_error("attention_fwd_long: unsupported (N, head_dim)");
    const auto [q, k, v] = qkv_operands(qkv, ld_qkv, B, N, H, hd);
    AttnFwdLongParams p;
    p.N = N, p.H = H, p.B = B, p.D = H * hd;
    p.scale_log2 = 1.4426950408889634f / sqrtf(static_cast<float>(hd));
    p.out = out, p.lse = lse;
    if (hd == 64) launch_fwd_long<64>(q, k, v, p, stream);
    else if (hd == 128) launch_fwd_long<128>(q, k, v, p, stream);
    else launch_fwd_long<160>(q, k, v, p, stream);
}

void attention_bwd(const __nv_bfloat16* qkv, int64_t ld_qkv, const __nv_bfloat16* dout, int64_t ld_do,
                   const __nv_bfloat16* out, int64_t ld_o, const float* lse, float* delta, __nv_bfloat16* dqkv,
                   int B, int N, int H, int hd, cudaStream_t stream, bool persist, float* colsum) {
    if (!attention_bwd_supported(N, hd)) throw std::runtime_error("attention_bwd: unsupported (N, head_dim)");
    const int D = H * hd;
    {
        const int64_t threads = static_cast<int64_t>(B) * N * H * 4;
        // persist: `delta` holds two [B*H, N] planes -- delta, then lse * log2(e)
        float* lse2 = persist ? delta + static_cast<int64_t>(B) * H * N : nullptr;
        attn_delta_kernel<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, stream>>>(dout, ld_do, out, ld_o, delta,
                                                                                           lse, lse2, B, N, H, hd);
        cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess) throw std::runtime_error(std::string("attention delta launch: ") + cudaGetErrorString(err));
    }
    if (persist) {
        attention_bwd_persist_core(qkv, ld_qkv, dout, ld_do, delta + static_cast<int64_t>(B) * H * N, delta, dqkv, colsum,
                                   B, N, H, hd, stream);
        return;
    }
    if (colsum != nullptr) throw std::runtime_error("attention_bwd: fused column sums need the persistent kernels");
    const auto [q, k, v] = qkv_operands(qkv, ld_qkv, B, N, H, hd);
    const GemmOperand dO = head_operand(dout, ld_do, B, N, H, hd);
    AttnBwdParams p;
    p.N = N, p.H = H, p.B = B, p.D = D;
    p.scale = 1.0f / sqrtf(static_cast<float>(hd));
    p.scale_log2 = p.scale * 1.4426950408889634f;
    p.lse = lse, p.delta = delta;
    p.out1 = p.out2 = nullptr;
    p.ld_out = 3 * static_cast<int64_t>(D);
    if (hd == 64) run_bwd<64>(q, k, v, dO, p, dqkv, stream);
    else if (hd == 128) run_bwd<128>(q, k, v, dO, p, dqkv, stream);
    else run_bwd<160>(q, k, v, dO, p, dqkv, stream);
}

}  // namespace b200
