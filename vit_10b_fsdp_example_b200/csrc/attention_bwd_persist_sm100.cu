// Persistent variant of the fused attention backward (attention_bwd_sm100.cu) for sm_100a.
//
// Same math, same two roles (kT = true: a CTA owns 128 keys and produces dK / dV; kT = false: a CTA owns 128 queries
// and produces dQ), same TMA / tcgen05 operand layouts.  What changes is the schedule, aimed at the hd = 160 case
// where only one CTA fits an SM and the one-shot kernel spends ~40 % of its 13.5 us per CTA outside the tile pipeline
// (launch + barrier / TMEM setup, the first resident-tile load, the first score MMA, the epilogue):
//   * one CTA per SM stays alive and loops over work items (image, head, 128-row block); the Y-tile ring, the T_s / T_p
//     buffers and the P / dS staging buffers simply keep cycling across item boundaries;
//   * the resident tiles of item i+1 are requested as soon as the last score MMA of item i has drained them, so that
//     load, the first score MMA of item i+1 and the epilogue of item i overlap;
//   * EIGHT softmax warps (two per TMEM lane quarter, each taking 32 of a tile's 64 columns) halve the per-tile
//     exp2 / dS critical path, and the epilogue columns are split the same way;
//   * the epilogue goes through a SWIZZLE_64B staging tile and a TMA store per 32-column chunk (the forward's
//     in-kernel timeline showed per-thread 16-byte stores to 32 scattered rows costing ~900 cycles per chunk), and the
//     qkv bias gradient (column sums of dq / dk / dv) is reduced from that staging tile instead of re-reading the
//     1 GB dqkv tensor with a separate kernel;
//   * key / query masks are compiled out when N is a multiple of 128.
// Instantiated for hd = 160 only; chosen there when N % 4 == 0 (ops/attention_plan.py).
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

long long* g_bwd_trace = nullptr;  // optional in-kernel timeline target (attention_bwd_set_trace)
int g_bwd_trace_tiles = 0;
int g_bwd_trace_role_v = 0;

constexpr int kThreads = 320;  // warp 0: TMA, warp 1: MMA + TMEM, warps 2-9: softmax-backward math + epilogue
constexpr int kTileC = 64;
constexpr int kMaxSeqP = 1024;

struct BwdPParams {
    int N, H, B, D;
    int nblk;   // 128-row blocks per (image, head)
    int total;  // work items
    float scale, scale_log2;
    const float* lse;    // [B*H, N] row log-sum-exp ALREADY in log2 units (written by attn_delta_kernel)
    const float* delta;  // [B*H, N] rowsum(dO o O)
    __nv_bfloat16* out1;
    __nv_bfloat16* out2;
    int64_t ld_out;
    float* colsum1;  // optional: fp32 column sums of out1 (qkv bias gradient slice), indexed h * hd + column
    float* colsum2;
    long long* trace;  // optional clock64 timeline of CTA 0 (16 slots per global tile index), see stampb()
    int trace_tiles;
};

// trace slots per tile: 0 producer issued Y, 1 MMA saw y_full + ts buffer free (T_s issue), 2 MMA T_p issue, 3 MMA got
// d_full (accumulate issue), 4 softmax saw ts_full, 5 softmax finished P, 6 softmax saw tp_full, 7 softmax finished dS,
// 8 epilogue start (last tile of an item), 9 epilogue end, 10 producer issued next X
__device__ __forceinline__ void stampb(const BwdPParams& p, int tile, int slot) {
    if (p.trace != nullptr && blockIdx.x == 0 && tile < p.trace_tiles) p.trace[tile * 16 + slot] = clock64();
}

__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

template <int HD, bool kT>
struct BwdPCfg {
    static constexpr int W = (HD % 64 == 0) ? 64 : 32;
    static constexpr int kAtoms = HD / W;
    static constexpr uint32_t kLayout = (W == 64) ? 2u : 4u;
    static constexpr int kRowBytes = W * 2;
    static constexpr int kXBytes = 128 * HD * 2;
    static constexpr int kYBytes = kTileC * HD * 2;
    static constexpr int kStageBytes = 2 * kYBytes;
    static constexpr int kEBytes = 128 * kTileC * 2;
    static constexpr int kTsBufs = 2;
    static constexpr int kNumAcc = kT ? 2 : 1;
    static constexpr int kColTs = 0;
    static constexpr int kColTp = kTsBufs * kTileC;
    static constexpr int kColAcc1 = kColTp + kTileC;
    static constexpr int kColAcc2 = kColAcc1 + HD;
    static constexpr int kColsUsed = kColAcc1 + kNumAcc * HD;
    static constexpr int kTmemCols = kColsUsed <= 256 ? 256 : 512;
    __host__ __device__ static constexpr int stat_bytes(int n_tokens) {
        return kT ? 2 * 2 * 4 * ((n_tokens + kTileC - 1) / kTileC) * kTileC : 0;  // 2 stages x (lse2 | delta)
    }
    static constexpr int kOBytes = 128 * 32 * 2;  // epilogue staging tile per warp group (128 rows x 32 columns)
    __host__ __device__ static constexpr int smem_bytes(int n_tokens) {
        return 2 * kXBytes + 2 * kStageBytes + 2 * kEBytes + 2 * kOBytes + stat_bytes(n_tokens) + 256;
    }
    static_assert(kColsUsed <= 512, "TMEM budget exceeded");
};

template <int HD, bool kT, bool kMask>
__global__ void __launch_bounds__(kThreads) attn_bwd_persist_sm100_kernel(const __grid_constant__ CUtensorMap tmap_x1,
                                                                         const __grid_constant__ CUtensorMap tmap_x2,
                                                                         const __grid_constant__ CUtensorMap tmap_y1,
                                                                         const __grid_constant__ CUtensorMap tmap_y2,
                                                                         const __grid_constant__ CUtensorMap tmap_o1,
                                                                         const __grid_constant__ CUtensorMap tmap_o2,
                                                                         const BwdPParams p) {
    using C = BwdPCfg<HD, kT>;
    constexpr int W = C::W, kAtoms = C::kAtoms, kRowBytes = C::kRowBytes, kTsBufs = C::kTsBufs;
    constexpr uint32_t kLayout = C::kLayout;
    constexpr uint32_t kSbo = 8 * kRowBytes;

    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sX1 = smem;
    uint8_t* sX2 = sX1 + C::kXBytes;
    uint8_t* sY = sX2 + C::kXBytes;
    uint8_t* sE = sY + 2 * C::kStageBytes;
    uint8_t* sD = sE + C::kEBytes;
    uint8_t* sO = sD + C::kEBytes;   // [2 warp groups] epilogue staging tiles
    const int nt = (p.N + kTileC - 1) / kTileC;
    // column statistics of the dK/dV role (per query: lse2, delta), bulk-copied by the producer, 2 stages
    float* s_stat = reinterpret_cast<float*>(sO + 2 * C::kOBytes);  // [stage][lse2 (nt*64) | delta (nt*64)]
    const int stat_stride = 2 * nt * kTileC;
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(s_stat) + C::stat_bytes(p.N));
    uint64_t* x_full = bars;
    uint64_t* x_empty = bars + 1;
    uint64_t* y_full = bars + 2;     // [2]
    uint64_t* y_empty = bars + 4;    // [2]
    uint64_t* ts_full = bars + 6;    // [2]
    uint64_t* ts_empty = bars + 8;   // [2]
    uint64_t* tp_full = bars + 10;
    uint64_t* tp_empty = bars + 11;
    uint64_t* e_full = bars + 12;
    uint64_t* e_empty = bars + 13;
    uint64_t* d_full = bars + 14;
    uint64_t* d_empty = bars + 15;
    uint64_t* acc_full = bars + 16;
    uint64_t* acc_empty = bars + 17;
    uint64_t* stat_full = bars + 18;   // [2]
    uint64_t* stat_empty = bars + 20;  // [2]
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 22);

    const uint32_t warp_idx = threadIdx.x / 32;
    const uint32_t lane = lane_id();
    const int n_items =
        (p.total - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
    const int n_tiles = n_items * nt;
    auto decode = [&](int i, int& blk, int& h, int& b) {
        const int w = static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x);
        blk = w % p.nblk;
        const int bh = w / p.nblk;
        h = bh % p.H;
        b = bh / p.H;
    };

    if (warp_idx == 0 && elect_one()) {
        prefetch_tmap(&tmap_x1);
        prefetch_tmap(&tmap_x2);
        prefetch_tmap(&tmap_y1);
        prefetch_tmap(&tmap_y2);
        prefetch_tmap(&tmap_o1);
        if constexpr (kT) prefetch_tmap(&tmap_o2);
        mbar_init(x_full, 1);
        mbar_init(x_empty, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&y_full[i], 1);
            mbar_init(&y_empty[i], 1);
            mbar_init(&ts_full[i], 1);
            mbar_init(&ts_empty[i], 8);
        }
        mbar_init(tp_full, 1);
        mbar_init(tp_empty, 8);
        mbar_init(e_full, 8);
        mbar_init(e_empty, 1);
        mbar_init(d_full, 8);
        mbar_init(d_empty, 1);
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, 8);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&stat_full[i], 1);
            mbar_init(&stat_empty[i], 8);
        }
        fence_mbar_init();
    }
    if (warp_idx == 1) tmem_alloc<1>(tmem_ptr_smem, C::kTmemCols);
    if constexpr (kT && kMask) {  // pad columns (queries >= N) are never bulk-copied: keep them finite
        for (int q = threadIdx.x; q < 2 * stat_stride; q += kThreads) s_stat[q] = 0.f;
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp_idx == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            auto load_x = [&](int i) {
                int blk, h, b;
                decode(i, blk, h, b);
                if constexpr (kT) {  // the item's per-query statistics ride along as two 1-D bulk copies
                    const int sg = i & 1;
                    if (i >= 2) mbar_wait(&stat_empty[sg], ((i >> 1) - 1) & 1);
                    const int64_t off = (static_cast<int64_t>(b) * p.H + h) * p.N;
                    float* dst = s_stat + sg * stat_stride;
                    mbar_arrive_expect_tx(&stat_full[sg], 2 * p.N * 4);
                    bulk_load_1d(dst, p.lse + off, p.N * 4, &stat_full[sg]);
                    bulk_load_1d(dst + nt * kTileC, p.delta + off, p.N * 4, &stat_full[sg]);
                }
                mbar_arrive_expect_tx(x_full, 2 * C::kXBytes);
#pragma unroll
                for (int a = 0; a < kAtoms; ++a) {
                    tma_load_4d(&tmap_x1, x_full, sX1 + a * (128 * kRowBytes), a * W, blk * 128, h, b);
                    tma_load_4d(&tmap_x2, x_full, sX2 + a * (128 * kRowBytes), a * W, blk * 128, h, b);
                }
            };
            if (n_items > 0) load_x(0);
            for (int t = 0; t < n_tiles; ++t) {
                const int i = t / nt, j = t - i * nt, st = t & 1;
                int blk, h, b;
                decode(i, blk, h, b);
                if (t >= 2) mbar_wait(&y_empty[st], ((t >> 1) - 1) & 1);
                uint8_t* y1 = sY + st * C::kStageBytes;
                uint8_t* y2 = y1 + C::kYBytes;
                mbar_arrive_expect_tx(&y_full[st], C::kStageBytes);
#pragma unroll
                for (int a = 0; a < kAtoms; ++a) {
                    tma_load_4d(&tmap_y1, &y_full[st], y1 + a * (kTileC * kRowBytes), a * W, j * kTileC, h, b);
                    tma_load_4d(&tmap_y2, &y_full[st], y2 + a * (kTileC * kRowBytes), a * W, j * kTileC, h, b);
                }
                stampb(p, t, 0);
                if (j == nt - 1 && i + 1 < n_items) {
                    // resident tiles of the next item: free once the last score MMAs of this item have read them
                    mbar_wait(x_empty, i & 1);
                    load_x(i + 1);
                    stampb(p, t, 10);
                }
            }
        }
    } else if (warp_idx == 1) {
        // ===================================== MMA issuer =====================================
        if (elect_one()) {
            constexpr uint32_t idesc_t = make_idesc_bf16(128, kTileC, 0, 0);
            constexpr uint32_t idesc_a = make_idesc_bf16(128, HD, 0, 1);
            auto issue_scores = [&](uint32_t tmem_d, const uint8_t* sx, const uint8_t* sy) {
#pragma unroll
                for (int k = 0; k < HD / 16; ++k) {
                    const int atom = (k * 16) / W, within = (k * 16) % W;
                    const uint64_t da = make_smem_desc(smem_u32(sx) + atom * (128 * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    const uint64_t db = make_smem_desc(smem_u32(sy) + atom * (kTileC * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    umma_bf16<1>(tmem_d, da, db, idesc_t, k > 0 ? 1u : 0u);
                }
            };
            auto issue_acc = [&](uint32_t tmem_d, const uint8_t* se, const uint8_t* sy, bool accumulate) {
#pragma unroll
                for (int k = 0; k < kTileC / 16; ++k) {
                    const uint64_t da = make_smem_desc(smem_u32(se) + k * 32, 0, 1024, 2u);
                    const uint64_t db = make_smem_desc(smem_u32(sy) + k * 16 * kRowBytes, kTileC * kRowBytes, kSbo, kLayout);
                    umma_bf16<1>(tmem_d, da, db, idesc_a, (accumulate || k > 0) ? 1u : 0u);
                }
            };
            // score tile T_s of global tile t1 (waits for its operands and for a free T_s buffer)
            auto prefetch_ts = [&](int t1) {
                const int i1 = t1 / nt, j1 = t1 - i1 * nt, s1 = t1 & 1, tb1 = t1 % kTsBufs;
                if (j1 == 0) mbar_wait(x_full, i1 & 1);
                mbar_wait(&y_full[s1], (t1 >> 1) & 1);
                if (t1 >= kTsBufs) mbar_wait(&ts_empty[tb1], (t1 / kTsBufs - 1) & 1);
                tc_fence_after();
                stampb(p, t1, 1);
                issue_scores(tmem_base + C::kColTs + tb1 * kTileC, sX1, sY + s1 * C::kStageBytes);
                umma_commit<1>(&ts_full[tb1]);
            };
            if (n_tiles > 0) prefetch_ts(0);
            for (int t = 0; t < n_tiles; ++t) {
                const int i = t / nt, j = t - i * nt, st = t & 1;
                const uint8_t* y1 = sY + st * C::kStageBytes;
                const uint8_t* y2 = y1 + C::kYBytes;
                const bool last_of_item = j == nt - 1;
                if (t > 0) mbar_wait(tp_empty, (t - 1) & 1);
                tc_fence_after();
                stampb(p, t, 2);
                issue_scores(tmem_base + C::kColTp, sX2, y2);
                umma_commit<1>(tp_full);
                if (last_of_item) umma_commit<1>(x_empty);  // both score MMAs of the item's last tile are issued
                // next score tile of the SAME item goes first (it runs under this tile's exponentials); across an
                // item boundary it would block on the next resident-tile load, so there the accumulation goes first
                if (!last_of_item && t + 1 < n_tiles) prefetch_ts(t + 1);
                if (j == 0 && i > 0) mbar_wait(acc_empty, (i - 1) & 1);  // previous item's epilogue has read O
                if constexpr (kT) {
                    mbar_wait(e_full, t & 1);
                    tc_fence_after();
                    issue_acc(tmem_base + C::kColAcc2, sE, y2, j > 0);
                    umma_commit<1>(e_empty);
                }
                mbar_wait(d_full, t & 1);
                tc_fence_after();
                stampb(p, t, 3);
                issue_acc(tmem_base + C::kColAcc1, sD, y1, j > 0);
                umma_commit<1>(d_empty);
                umma_commit<1>(&y_empty[st]);
                if (last_of_item) {
                    umma_commit<1>(acc_full);
                    if (t + 1 < n_tiles) prefetch_ts(t + 1);
                }
            }
        }
    } else {
        // ============================ softmax-backward math + epilogue (8 warps) ============================
        const uint32_t quarter = warp_idx & 3;
        const uint32_t grp = (warp_idx - 2) >> 2;        // which 32-column half of every tile
        const uint32_t r = quarter * 32 + lane;
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16);
        constexpr float kLog2e = 1.4426950408889634f;
        const uint32_t erow = smem_u32(sE) + r * 128;
        const uint32_t drow = smem_u32(sD) + r * 128;
        const int tid = static_cast<int>(threadIdx.x) - 64;  // 0 .. 255
        for (int i = 0; i < n_items; ++i) {
            int blk, h, b;
            decode(i, blk, h, b);
            const int64_t bh = static_cast<int64_t>(b) * p.H + h;
            const int row = blk * 128 + static_cast<int>(r);
            const bool row_ok = row < p.N;
            float lse2_r = 0.f, delta_r = 0.f;
            const float* s_lse2 = s_stat + (i & 1) * stat_stride;
            const float* s_delta = s_lse2 + nt * kTileC;
            if constexpr (kT) {
                mbar_wait(&stat_full[i & 1], (i >> 1) & 1);  // landed long ago: requested with the resident tiles
            } else {
                if (row_ok) {
                    lse2_r = p.lse[bh * p.N + row];
                    delta_r = p.delta[bh * p.N + row];
                }
            }
            for (int j = 0; j < nt; ++j) {
                const int t = i * nt + j, tb = t % kTsBufs;
                const int col0 = j * kTileC + static_cast<int>(grp) * 32;
                uint32_t pk[16];
                mbar_wait(&ts_full[tb], (t / kTsBufs) & 1);
                if (warp_idx == 2 && lane == 0) stampb(p, t, 4);
                tc_fence_after();
                if constexpr (kT) {
                    if (t > 0) mbar_wait(e_empty, (t - 1) & 1);
                }
                {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(taddr + C::kColTs + tb * kTileC + grp * 32, v);
                    float lcol[32];
                    if constexpr (kT) {  // 8 x LDS.128 (warp-wide broadcast) instead of 32 scalar loads
#pragma unroll
                        for (int x = 0; x < 32; x += 4) {
                            const float4 l4 = *reinterpret_cast<const float4*>(s_lse2 + col0 + x);
                            lcol[x] = l4.x, lcol[x + 1] = l4.y, lcol[x + 2] = l4.z, lcol[x + 3] = l4.w;
                        }
                    }
                    tmem_ld_wait();
#pragma unroll
                    for (int x = 0; x < 32; x += 2) {
                        const int col = col0 + x;
                        float l0, l1;
                        if constexpr (kT) {
                            l0 = lcol[x], l1 = lcol[x + 1];
                        } else {
                            l0 = l1 = lse2_r;
                        }
                        float e0 = exp2f(fmaf(__uint_as_float(v[x]), p.scale_log2, -l0));
                        float e1 = exp2f(fmaf(__uint_as_float(v[x + 1]), p.scale_log2, -l1));
                        if (kMask) {
                            e0 = (row_ok && col < p.N) ? e0 : 0.f;
                            e1 = (row_ok && col + 1 < p.N) ? e1 : 0.f;
                        }
                        pk[x / 2] = pack_bf16x2(e0, e1);
                    }
                    if constexpr (kT) {
#pragma unroll
                        for (int j8 = 0; j8 < 4; ++j8) {
                            const uint32_t chunk = grp * 4 + j8;
                            st_shared_v4(erow + ((chunk ^ (r & 7)) << 4), pk[j8 * 4], pk[j8 * 4 + 1], pk[j8 * 4 + 2],
                                         pk[j8 * 4 + 3]);
                        }
                    }
                }
                tc_fence_before();
                if constexpr (kT) fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&ts_empty[tb]);
                    if constexpr (kT) mbar_arrive(e_full);
                }

                if (warp_idx == 2 && lane == 0) stampb(p, t, 5);
                mbar_wait(tp_full, t & 1);
                if (warp_idx == 2 && lane == 0) stampb(p, t, 6);
                tc_fence_after();
                if (t > 0) mbar_wait(d_empty, (t - 1) & 1);
                {
                    uint32_t v[32];
                    tmem_ld_32x32b_x32(taddr + C::kColTp + grp * 32, v);
                    float dcol[32];
                    if constexpr (kT) {
#pragma unroll
                        for (int x = 0; x < 32; x += 4) {
                            const float4 d4 = *reinterpret_cast<const float4*>(s_delta + col0 + x);
                            dcol[x] = d4.x, dcol[x + 1] = d4.y, dcol[x + 2] = d4.z, dcol[x + 3] = d4.w;
                        }
                    }
                    tmem_ld_wait();
                    uint32_t dk[16];
#pragma unroll
                    for (int x = 0; x < 32; x += 2) {
                        float d0, d1;
                        if constexpr (kT) {
                            d0 = dcol[x], d1 = dcol[x + 1];
                        } else {
                            d0 = d1 = delta_r;
                        }
                        const uint32_t pw = pk[x / 2];
                        const float s0 = bf16_lo(pw) * (__uint_as_float(v[x]) - d0) * p.scale;
                        const float s1 = bf16_hi(pw) * (__uint_as_float(v[x + 1]) - d1) * p.scale;
                        dk[x / 2] = pack_bf16x2(s0, s1);
                    }
#pragma unroll
                    for (int j8 = 0; j8 < 4; ++j8) {
                        const uint32_t chunk = grp * 4 + j8;
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
                if (warp_idx == 2 && lane == 0) stampb(p, t, 7);
            }

            if constexpr (kT) {  // this warp no longer reads the item's statistics stage
                __syncwarp();
                if (lane == 0) mbar_arrive(&stat_empty[i & 1]);
            }
            // ---- epilogue of item i: the two warp groups take alternating 32-column chunks; every chunk goes
            //      TMEM -> bf16 -> SWIZZLE_64B staging tile of the group -> TMA store (rows beyond the image are
            //      clipped by the tensor map) and, from the same tile, into the bias-gradient column sums ----
            mbar_wait(acc_full, i & 1);
            if (warp_idx == 2 && lane == 0) stampb(p, i * nt + nt - 1, 8);
            tc_fence_after();
            // two staging tiles per warp group: its slice of sO and -- idle during the epilogue -- its slice of the P tile
            uint8_t* const obufs[2] = {sO + grp * C::kOBytes, sE + grp * C::kOBytes};
            uint32_t flip = 0;
            const uint32_t gtid = (threadIdx.x - 64) & 127;  // thread index inside the warp group
#pragma unroll
            for (int a = 0; a < C::kNumAcc; ++a) {
                const uint32_t cbase = (a == 0) ? C::kColAcc1 : C::kColAcc2;
                float* csum = (a == 0) ? p.colsum1 : p.colsum2;
#pragma unroll 1
                for (int c = static_cast<int>(grp); c < HD / 32; c += 2) {
                    uint32_t v[32];
                    uint8_t* obuf = obufs[flip & 1];
                    ++flip;
                    tmem_ld_32x32b_x32(taddr + cbase + c * 32, v);
                    if (gtid == 0) tma_store_wait_read<1>();  // the store that last read this tile has drained it
                    named_bar_sync(2 + grp, 128);
                    tmem_ld_wait();
                    const uint32_t orow = smem_u32(obuf) + r * 64;
                    uint32_t pk[16];
#pragma unroll
                    for (int x = 0; x < 16; ++x)
                        pk[x] = pack_bf16x2(__uint_as_float(v[2 * x]), __uint_as_float(v[2 * x + 1]));
#pragma unroll
                    for (int j8 = 0; j8 < 4; ++j8)
                        st_shared_v4(orow + ((j8 ^ ((r >> 1) & 3)) << 4), pk[j8 * 4], pk[j8 * 4 + 1], pk[j8 * 4 + 2],
                                     pk[j8 * 4 + 3]);
                    fence_proxy_async_smem();
                    named_bar_sync(2 + grp, 128);
                    if (gtid == 0) {
                        if (a == 0) tma_store_4d(&tmap_o1, obuf, c * 32, blk * 128, h, b);
                        else tma_store_4d(&tmap_o2, obuf, c * 32, blk * 128, h, b);
                        tma_store_commit();
                    }
                    if (csum != nullptr) {
                        // Column sums of this warp's 32 rows (the bf16 values that were stored) by a butterfly
                        // transpose-reduce over the lanes: 31 shuffles for all 32 columns; lane l ends with column l.
                        float cv[32];
#pragma unroll
                        for (int x = 0; x < 16; ++x) {
                            cv[2 * x] = bf16_lo(pk[x]);
                            cv[2 * x + 1] = bf16_hi(pk[x]);
                        }
#pragma unroll
                        for (int sft = 16; sft >= 1; sft >>= 1) {
                            const bool upper = (lane & sft) != 0;
#pragma unroll
                            for (int k = 0; k < sft; ++k) {
                                const float send = upper ? cv[k] : cv[k + sft];
                                const float keep = upper ? cv[k + sft] : cv[k];
                                cv[k] = keep + __shfl_xor_sync(0xffffffffu, send, sft);
                            }
                        }
                        atomicAdd(csum + h * HD + c * 32 + lane, cv[0]);
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty);
            // the P tile doubles as staging for BOTH groups (rows 0-63 / 64-127) while the next item's P writes of either
            // group cover all 128 rows: every store must have read its tile before any of the 8 warps moves on
            if (gtid == 0) tma_store_wait_read<0>();
            named_bar_sync(1, 256);
            if (warp_idx == 2 && lane == 0) stampb(p, i * nt + nt - 1, 9);
        }
        if (((threadIdx.x - 64) & 127) == 0) tma_store_wait<0>();
    }
    __syncthreads();
    if (warp_idx == 1) tmem_dealloc<1>(tmem_base, C::kTmemCols);
}

template <int HD, bool kT, bool kMask>
void launch_bwd_persist(const GemmOperand& x1, const GemmOperand& x2, const GemmOperand& y1, const GemmOperand& y2,
                        const GemmOperand& o1, const GemmOperand& o2, const BwdPParams& p, cudaStream_t stream) {
    using C = BwdPCfg<HD, kT>;
    if (C::smem_bytes(p.N) > 232448) throw std::runtime_error("attention bwd-persist: sequence too long for shared memory");
    auto kern = attn_bwd_persist_sm100_kernel<HD, kT, kMask>;
    static bool attr_set = false;
    static int num_sms = 0;
    if (!attr_set) {
        cudaError_t err =
            cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 C::smem_bytes(kMaxSeqP) > 232448 ? 232448 : C::smem_bytes(kMaxSeqP));
        if (err != cudaSuccess)
            throw std::runtime_error(std::string("attention bwd-persist smem attr: ") + cudaGetErrorString(err));
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        attr_set = true;
    }
    const int sw = C::W * 2;
    CUtensorMap tx1 = make_tensor_map_4d(x1, HD, p.N, C::W, 128, sw);
    CUtensorMap tx2 = make_tensor_map_4d(x2, HD, p.N, C::W, 128, sw);
    CUtensorMap ty1 = make_tensor_map_4d(y1, HD, p.N, C::W, kTileC, sw);
    CUtensorMap ty2 = make_tensor_map_4d(y2, HD, p.N, C::W, kTileC, sw);
    CUtensorMap to1 = make_tensor_map_4d(o1, HD, p.N, 32, 128, 64);  // store boxes: 32 columns x 128 rows, SWIZZLE_64B
    CUtensorMap to2 = make_tensor_map_4d(kT ? o2 : o1, HD, p.N, 32, 128, 64);
    const int grid = p.total < num_sms ? p.total : num_sms;
    kern<<<grid, kThreads, C::smem_bytes(p.N), stream>>>(tx1, tx2, ty1, ty2, to1, to2, p);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess)
        throw std::runtime_error(std::string("attention bwd-persist launch: ") + cudaGetErrorString(err));
}

template <int HD>
void run_bwd_persist(const GemmOperand& q, const GemmOperand& k, const GemmOperand& v, const GemmOperand& dO,
                     BwdPParams p, __nv_bfloat16* dqkv, float* colsum, cudaStream_t stream) {
    // dq / dk / dv slices of dqkv viewed as [B][H][N rows, hd columns]: what the epilogue's TMA stores address
    const auto [oq, ok, ov] = qkv_operands(dqkv, p.ld_out, p.B, p.N, p.H, HD);
    const bool mask = p.N % 128 != 0;
    p.out1 = dqkv + p.D, p.out2 = dqkv + 2 * p.D;
    p.colsum1 = colsum != nullptr ? colsum + p.D : nullptr;
    p.colsum2 = colsum != nullptr ? colsum + 2 * p.D : nullptr;
    long long* const tr = p.trace;
    p.trace = g_bwd_trace_role_v == 0 ? tr : nullptr;
    if (mask) launch_bwd_persist<HD, true, true>(k, v, q, dO, ok, ov, p, stream);   // dK, dV
    else launch_bwd_persist<HD, true, false>(k, v, q, dO, ok, ov, p, stream);
    p.out1 = dqkv, p.out2 = nullptr;
    p.colsum1 = colsum, p.colsum2 = nullptr;
    p.trace = g_bwd_trace_role_v == 1 ? tr : nullptr;
    if (mask) launch_bwd_persist<HD, false, true>(q, dO, k, v, oq, oq, p, stream);  // dQ
    else launch_bwd_persist<HD, false, false>(q, dO, k, v, oq, oq, p, stream);
}

}  // namespace

// Optional in-kernel timeline (SURVEY 5.1): role 0 = dK/dV kernel, 1 = dQ kernel write into the same buffer layout
// (the dQ launch overwrites the dK/dV stamps unless trace_role selects one).
void attention_bwd_set_trace(long long* buf, int tiles, int role) {
    g_bwd_trace = buf, g_bwd_trace_tiles = tiles, g_bwd_trace_role_v = role;
}

// delta must already hold rowsum(dO o O) (attention_bwd computes it; see attention_bwd_sm100.cu)
void attention_bwd_persist_core(const __nv_bfloat16* qkv, int64_t ld_qkv, const __nv_bfloat16* dout, int64_t ld_do,
                                const float* lse, const float* delta, __nv_bfloat16* dqkv, float* colsum, int B, int N,
                                int H, int hd, cudaStream_t stream) {
    // instantiated for hd = 160 only: where two one-shot CTAs fit an SM (hd <= 128) those win; the per-row
    // statistics are bulk-copied in 16-byte units
    if (hd != 160 || N % 4 != 0) throw std::runtime_error("attention_bwd_persist: unsupported (N, head_dim)");
    const int D = H * hd;
    const auto [q, k, v] = qkv_operands(qkv, ld_qkv, B, N, H, hd);
    const GemmOperand dO = head_operand(dout, ld_do, B, N, H, hd);
    BwdPParams p;
    p.N = N, p.H = H, p.B = B, p.D = D;
    p.nblk = (N + 127) / 128;
    p.total = B * H * p.nblk;
    p.scale = 1.0f / sqrtf(static_cast<float>(hd));
    p.scale_log2 = p.scale * 1.4426950408889634f;
    p.lse = lse, p.delta = delta;
    p.out1 = p.out2 = nullptr;
    p.colsum1 = p.colsum2 = nullptr;
    p.trace = g_bwd_trace, p.trace_tiles = g_bwd_trace_tiles;
    p.ld_out = 3 * static_cast<int64_t>(D);
    run_bwd_persist<160>(q, k, v, dO, p, dqkv, colsum, stream);
}

}  // namespace b200
