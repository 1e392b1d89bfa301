// Persistent, software-pipelined attention forward for sm_100a (128 < N <= 256 tokens, head dim 160).
//
// The one-shot kernel in attention_sm100.cu runs load -> S MMA -> softmax -> PV MMA -> store strictly in sequence and
// only one CTA fits an SM at hd = 160 (200 KB of shared memory), so nothing hides its loads (ncu: tensor pipe 9 %,
// DRAM 21 %, 773 us against a 210 us DRAM floor; profiles/r1e_attention_fwd_fused.md).  This kernel keeps ONE CTA per
// SM alive for the whole launch and lets its warps run ahead across work items (image, head, 128-query block):
//   warp 0   TMA producer: Q + K of item i+1 are requested as soon as the S MMAs of item i have drained them; V is
//            streamed in 64-key tiles through a 2-stage ring;
//   warp 1   tcgen05.mma issuer: S = Q K^T (N = 256) for item i+1 is issued right after the PV MMAs of item i, i.e. it
//            runs under the epilogue of item i;  O += P_j V_j per 64-key tile as soon as that tile of P is staged;
//   warps 2-5 softmax, one thread per query row: row max, exp2, un-normalised bf16 P into a 2-deep shared-memory ring
//            (K-major SWIZZLE_128B, the A operand of the PV MMA), log-sum-exp; key-column masks are compiled out when
//            N is a multiple of 64 (ViT-10B: 256);
//   warps 6-9 epilogue, one thread per query row: O from TMEM x 1/sum -> bf16 -> SWIZZLE_64B staging tile -> TMA store
//            (coalesced, clipped at the image boundary by the tensor map); it runs under the softmax of the NEXT item.
// The in-kernel timeline (clock64 stamps, tools/exp_ln_trace.py) of the first version -- softmax and epilogue on the
// same four warps, per-thread 16-byte global stores -- showed where an item's 16.5 K cycles went: pass 2 (exp2 + pack,
// masks on every element) 8.4 K, epilogue 4.6 K (32 scattered rows per store instruction), pass 1 1.7 K, waits 1.8 K;
// tensor pipe and TMA were idle most of the time.  Hence the split roles, the TMA store and the mask-free fast path.
// TMEM: S [128 x 256] fp32 + O [128 x hd] fp32 (416 columns at hd = 160).  Shared memory: Q 40 KB + K 80 KB +
// V ring 40 KB + P ring 32 KB + O staging 16 KB = 208 KB at hd = 160.  Scores never reach HBM.
// Replaces timm Attention's materialised softmax (reference run_vit_training.py:134 -> timm Block -> Attention).
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

constexpr int kPThreads = 320;  // warp 0 TMA, warp 1 MMA, warps 2-5 softmax, warps 6-9 epilogue
constexpr int kVT = 64;    // keys per V / P tile
constexpr int kNK = 256;   // key columns of the score tile (padded)

struct PersistParams {
    int N, H, B, D;
    int nq;          // 128-query blocks per (image, head)
    int nkt;         // 64-key tiles per item
    int total;       // work items = B * H * nq
    float scale_log2, scale;
    __nv_bfloat16* out;
    float* lse;      // optional
    long long* trace;  // optional in-kernel timeline of CTA 0: clock64 stamps, 16 slots per work item (see kTr*)
    int trace_items;
};

// trace slots (per item): who / what
enum { kTrQkIssued = 0, kTrQkFull = 1, kTrSIssue = 2, kTrAccEmpty = 3, kTrPv0 = 4, kTrSFull = 8, kTrPass1 = 9,
       kTrPass2 = 10, kTrAccFull = 11, kTrEpiDone = 12 };
__device__ __forceinline__ void stamp(const PersistParams& p, int item, int slot) {
    if (p.trace != nullptr && blockIdx.x == 0 && item < p.trace_items) p.trace[item * 16 + slot] = clock64();
}

template <int HD>
struct PersistCfg {
    static constexpr int W = (HD % 64 == 0) ? 64 : 32;
    static constexpr int kAtoms = HD / W;
    static constexpr uint32_t kLayout = (W == 64) ? 2u : 4u;
    static constexpr int kRowBytes = W * 2;
    static constexpr int kQBytes = 128 * HD * 2;
    static constexpr int kKBytes = kNK * HD * 2;
    static constexpr int kVBytes = kVT * HD * 2;
    static constexpr int kEBytes = 128 * kVT * 2;
    static constexpr int kColAcc = kNK;
    static constexpr int kOBytes = 128 * 32 * 2;  // output staging tile: 128 rows x 32 columns (SWIZZLE_64B)
    static constexpr int kSmem = kQBytes + kKBytes + 2 * kVBytes + 2 * kEBytes + 2 * kOBytes + 2 * 128 * 4 + 256;
    static_assert(kNK + HD <= 512, "TMEM budget exceeded");
    static_assert(kSmem <= 232448, "shared memory budget exceeded");
};

template <int HD, bool kMask>
__global__ void __launch_bounds__(kPThreads) attn_fwd_persist_sm100_kernel(const __grid_constant__ CUtensorMap tmap_q,
                                                                          const __grid_constant__ CUtensorMap tmap_k,
                                                                          const __grid_constant__ CUtensorMap tmap_v,
                                                                          const __grid_constant__ CUtensorMap tmap_o,
                                                                          const PersistParams p) {
    using C = PersistCfg<HD>;
    constexpr int W = C::W, kAtoms = C::kAtoms, kRowBytes = C::kRowBytes;
    constexpr uint32_t kLayout = C::kLayout;
    constexpr uint32_t kSbo = 8 * kRowBytes;

    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sQ = smem;
    uint8_t* sK = sQ + C::kQBytes;
    uint8_t* sV = sK + C::kKBytes;               // [2 stages]
    uint8_t* sE = sV + 2 * C::kVBytes;           // [2 buffers]
    uint8_t* sO = sE + 2 * C::kEBytes;           // [2 buffers] output staging
    float* s_inv = reinterpret_cast<float*>(sO + 2 * C::kOBytes);  // [2 items][128 rows] 1 / row sum
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_inv + 2 * 128);
    uint64_t* qk_full = bars;
    uint64_t* qk_empty = bars + 1;
    uint64_t* s_full = bars + 2;
    uint64_t* s_empty = bars + 3;
    uint64_t* acc_full = bars + 4;
    uint64_t* acc_empty = bars + 5;
    uint64_t* v_full = bars + 6;    // [2]
    uint64_t* v_empty = bars + 8;   // [2]
    uint64_t* e_full = bars + 10;   // [2]
    uint64_t* e_empty = bars + 12;  // [2]
    uint64_t* stat_full = bars + 14;  // [2] softmax -> epilogue: 1/sum of the item's rows is in s_inv
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 16);

    const uint32_t warp_idx = threadIdx.x / 32;
    const uint32_t lane = lane_id();
    const int nkt = p.nkt;
    // static striding: neighbouring CTAs work on the two query blocks of the same (image, head) -> K / V hit in L2
    const int n_items = (p.total - static_cast<int>(blockIdx.x) + static_cast<int>(gridDim.x) - 1) / static_cast<int>(gridDim.x);
    auto decode = [&](int i, int& qb, int& h, int& b) {
        const int w = static_cast<int>(blockIdx.x) + i * static_cast<int>(gridDim.x);
        qb = w % p.nq;
        const int bh = w / p.nq;
        h = bh % p.H;
        b = bh / p.H;
    };

    if (warp_idx == 0 && elect_one()) {
        prefetch_tmap(&tmap_q);
        prefetch_tmap(&tmap_k);
        prefetch_tmap(&tmap_v);
        prefetch_tmap(&tmap_o);
        mbar_init(qk_full, 1);
        mbar_init(qk_empty, 1);
        mbar_init(s_full, 1);
        mbar_init(s_empty, 4);
        mbar_init(acc_full, 1);
        mbar_init(acc_empty, 4);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&v_full[i], 1);
            mbar_init(&v_empty[i], 1);
            mbar_init(&e_full[i], 4);
            mbar_init(&e_empty[i], 1);
            mbar_init(&stat_full[i], 4);
        }
        fence_mbar_init();
    }
    if (warp_idx == 1) tmem_alloc<1>(tmem_ptr_smem, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp_idx == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            auto load_qk = [&](int i) {
                int qb, h, b;
                decode(i, qb, h, b);
                mbar_arrive_expect_tx(qk_full, C::kQBytes + C::kKBytes);
#pragma unroll
                for (int a = 0; a < kAtoms; ++a) {
                    tma_load_4d(&tmap_q, qk_full, sQ + a * (128 * kRowBytes), a * W, qb * 128, h, b);
                    tma_load_4d(&tmap_k, qk_full, sK + a * (kNK * kRowBytes), a * W, 0, h, b);
                }
            };
            auto load_v = [&](int i, int j) {
                int qb, h, b;
                decode(i, qb, h, b);
                const int t = i * nkt + j, st = t & 1;
                if (t >= 2) mbar_wait(&v_empty[st], ((t >> 1) - 1) & 1);
                uint8_t* dst = sV + st * C::kVBytes;
                mbar_arrive_expect_tx(&v_full[st], C::kVBytes);
#pragma unroll
                for (int a = 0; a < kAtoms; ++a)
                    tma_load_4d(&tmap_v, &v_full[st], dst + a * (kVT * kRowBytes), a * W, j * kVT, h, b);
            };
            if (n_items > 0) load_qk(0);
            for (int i = 0; i < n_items; ++i) {
                const int first = nkt < 2 ? nkt : 2;
                for (int j = 0; j < first; ++j) load_v(i, j);
                if (i + 1 < n_items) {  // Q / K of the next item as soon as this item's S MMAs have drained them
                    mbar_wait(qk_empty, i & 1);
                    load_qk(i + 1);
                    stamp(p, i + 1, kTrQkIssued);
                }
                for (int j = first; j < nkt; ++j) load_v(i, j);
            }
        }
    } else if (warp_idx == 1) {
        // ===================================== MMA issuer =====================================
        if (elect_one()) {
            constexpr uint32_t idesc_s = make_idesc_bf16(128, kNK, 0, 0);
            constexpr uint32_t idesc_o = make_idesc_bf16(128, HD, 0, 1);
            for (int i = 0; i < n_items; ++i) {
                mbar_wait(qk_full, i & 1);
                stamp(p, i, kTrQkFull);
                if (i > 0) mbar_wait(s_empty, (i - 1) & 1);
                stamp(p, i, kTrSIssue);
                tc_fence_after();
#pragma unroll
                for (int k = 0; k < HD / 16; ++k) {
                    const int atom = (k * 16) / W, within = (k * 16) % W;
                    const uint64_t da = make_smem_desc(smem_u32(sQ) + atom * (128 * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    const uint64_t db = make_smem_desc(smem_u32(sK) + atom * (kNK * kRowBytes) + within * 2, 0, kSbo, kLayout);
                    umma_bf16<1>(tmem_base, da, db, idesc_s, k > 0 ? 1u : 0u);
                }
                umma_commit<1>(s_full);
                umma_commit<1>(qk_empty);
                if (i > 0) mbar_wait(acc_empty, (i - 1) & 1);
                stamp(p, i, kTrAccEmpty);
                for (int j = 0; j < nkt; ++j) {
                    const int t = i * nkt + j, st = t & 1;
                    mbar_wait(&v_full[st], (t >> 1) & 1);
                    mbar_wait(&e_full[st], (t >> 1) & 1);
                    if (j < 4) stamp(p, i, kTrPv0 + j);
                    tc_fence_after();
                    const uint8_t* se = sE + st * C::kEBytes;
                    const uint8_t* sv = sV + st * C::kVBytes;
#pragma unroll
                    for (int k = 0; k < kVT / 16; ++k) {
                        const uint64_t da = make_smem_desc(smem_u32(se) + k * 32, 0, 1024, 2u);
                        const uint64_t db = make_smem_desc(smem_u32(sv) + k * 16 * kRowBytes, kVT * kRowBytes, kSbo, kLayout);
                        umma_bf16<1>(tmem_base + C::kColAcc, da, db, idesc_o, (j > 0 || k > 0) ? 1u : 0u);
                    }
                    umma_commit<1>(&e_empty[st]);
                    umma_commit<1>(&v_empty[st]);
                }
                umma_commit<1>(acc_full);
            }
        }
    } else if (warp_idx < 6) {
        // ===================================== softmax (warps 2-5) =====================================
        const uint32_t quarter = warp_idx & 3;
        const uint32_t r = quarter * 32 + lane;
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16);
        for (int i = 0; i < n_items; ++i) {
            int qb, h, b;
            decode(i, qb, h, b);
            const int q = qb * 128 + static_cast<int>(r);
            const bool row_ok = q < p.N;
            mbar_wait(s_full, i & 1);
            if (warp_idx == 2 && lane == 0) stamp(p, i, kTrSFull);
            tc_fence_after();
            // ---- pass 1: row maximum ----
            float mx = -INFINITY;
            for (int c = 0; c < nkt; ++c) {
                uint32_t v0[32], v1[32];
                tmem_ld_32x32b_x32(taddr + c * 64, v0);
                tmem_ld_32x32b_x32(taddr + c * 64 + 32, v1);
                tmem_ld_wait();
#pragma unroll
                for (int x = 0; x < 32; ++x) {
                    if (!kMask || c * 64 + x < p.N) mx = fmaxf(mx, __uint_as_float(v0[x]));
                    if (!kMask || c * 64 + 32 + x < p.N) mx = fmaxf(mx, __uint_as_float(v1[x]));
                }
            }
            const float m_scaled = mx * p.scale_log2;
            float sum = 0.f;
            if (warp_idx == 2 && lane == 0) stamp(p, i, kTrPass1);
            // ---- pass 2: P = exp2(S * c - m) per 64-key tile -> shared memory ----
            for (int j = 0; j < nkt; ++j) {
                const int t = i * nkt + j, eb = t & 1;
                uint32_t v0[32], v1[32];
                tmem_ld_32x32b_x32(taddr + j * kVT, v0);
                tmem_ld_32x32b_x32(taddr + j * kVT + 32, v1);
                if (t >= 2) mbar_wait(&e_empty[eb], ((t >> 1) - 1) & 1);
                const uint32_t erow = smem_u32(sE) + eb * C::kEBytes + r * 128;
                tmem_ld_wait();
                uint32_t pk[32];
                float s0 = 0.f, s1 = 0.f;  // two independent accumulation chains
#pragma unroll
                for (int x = 0; x < 32; x += 2) {
                    const int col = j * kVT + x;
                    float e0 = exp2f(fmaf(__uint_as_float(v0[x]), p.scale_log2, -m_scaled));
                    float e1 = exp2f(fmaf(__uint_as_float(v0[x + 1]), p.scale_log2, -m_scaled));
                    float f0 = exp2f(fmaf(__uint_as_float(v1[x]), p.scale_log2, -m_scaled));
                    float f1 = exp2f(fmaf(__uint_as_float(v1[x + 1]), p.scale_log2, -m_scaled));
                    if (kMask) {
                        e0 = col < p.N ? e0 : 0.f;
                        e1 = col + 1 < p.N ? e1 : 0.f;
                        f0 = col + 32 < p.N ? f0 : 0.f;
                        f1 = col + 33 < p.N ? f1 : 0.f;
                    }
                    s0 += e0 + e1;
                    s1 += f0 + f1;
                    pk[x / 2] = pack_bf16x2(e0, e1);
                    pk[16 + x / 2] = pack_bf16x2(f0, f1);
                }
                sum += s0 + s1;
#pragma unroll
                for (int ch = 0; ch < 8; ++ch)
                    st_shared_v4(erow + ((ch ^ (r & 7)) << 4), pk[ch * 4], pk[ch * 4 + 1], pk[ch * 4 + 2], pk[ch * 4 + 3]);
                fence_proxy_async_smem();  // generic-proxy P writes -> async-proxy (tensor core) reads
                __syncwarp();
                if (lane == 0) mbar_arrive(&e_full[eb]);
            }
            tc_fence_before();
            s_inv[(i & 1) * 128 + r] = 1.0f / sum;
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(s_empty);          // S of the next item may overwrite the score columns
                mbar_arrive(&stat_full[i & 1]);  // the epilogue warps may read this item's 1 / sum
            }
            if (warp_idx == 2 && lane == 0) stamp(p, i, kTrPass2);
            const int64_t bh = static_cast<int64_t>(b) * p.H + h;
            if (p.lse != nullptr && row_ok) p.lse[bh * p.N + q] = mx * p.scale + __logf(sum);
        }
    } else {
        // ===================================== epilogue (warps 6-9) =====================================
        const uint32_t quarter = warp_idx & 3;
        const uint32_t r = quarter * 32 + lane;
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16);
        const uint32_t et = threadIdx.x - 192;
        uint32_t flip = 0;
        for (int i = 0; i < n_items; ++i) {
            int qb, h, b;
            decode(i, qb, h, b);
            mbar_wait(&stat_full[i & 1], (i >> 1) & 1);
            const float inv = s_inv[(i & 1) * 128 + r];
            mbar_wait(acc_full, i & 1);
            if (warp_idx == 6 && lane == 0) stamp(p, i, kTrAccFull);
            tc_fence_after();
#pragma unroll 1
            for (int c = 0; c < HD / 32; ++c) {
                uint8_t* buf = sO + (flip & 1) * C::kOBytes;
                uint32_t v[32];
                tmem_ld_32x32b_x32(taddr + C::kColAcc + c * 32, v);
                if (et == 0) tma_store_wait_read<1>();  // the store that last read this buffer has drained it
                named_bar_sync(2, 128);
                tmem_ld_wait();
                if (c == HD / 32 - 1) {  // O is in registers: the PV MMAs of the next item may overwrite it
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(acc_empty);
                }
                // staging tile: [128 rows x 64 B], SWIZZLE_64B (16-byte chunk index ^= (row >> 1) & 3)
                const uint32_t orow = smem_u32(buf) + r * 64;
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    st_shared_v4(orow + ((j8 ^ ((r >> 1) & 3)) << 4),
                                 pack_bf16x2(__uint_as_float(v[j8 * 8]) * inv, __uint_as_float(v[j8 * 8 + 1]) * inv),
                                 pack_bf16x2(__uint_as_float(v[j8 * 8 + 2]) * inv, __uint_as_float(v[j8 * 8 + 3]) * inv),
                                 pack_bf16x2(__uint_as_float(v[j8 * 8 + 4]) * inv, __uint_as_float(v[j8 * 8 + 5]) * inv),
                                 pack_bf16x2(__uint_as_float(v[j8 * 8 + 6]) * inv, __uint_as_float(v[j8 * 8 + 7]) * inv));
                }
                fence_proxy_async_smem();
                named_bar_sync(2, 128);
                if (et == 0) {  // rows beyond the image (N not a multiple of 128) are clipped by the tensor map
                    tma_store_4d(&tmap_o, buf, c * 32, qb * 128, h, b);
                    tma_store_commit();
                }
                ++flip;
            }
            if (warp_idx == 6 && lane == 0) stamp(p, i, kTrEpiDone);
        }
        if (et == 0) tma_store_wait<0>();
    }
    __syncthreads();
    if (warp_idx == 1) tmem_dealloc<1>(tmem_base, 512);
}

template <int HD, bool kMask>
void launch_persist(const GemmOperand& q, const GemmOperand& k, const GemmOperand& v, const GemmOperand& o,
                    const PersistParams& p, cudaStream_t stream) {
    using C = PersistCfg<HD>;
    auto kern = attn_fwd_persist_sm100_kernel<HD, kMask>;
    static bool attr_set = false;
    static int num_sms = 0;
    if (!attr_set) {
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmem);
        if (err != cudaSuccess)
            throw std::runtime_error(std::string("attention persist smem attr: ") + cudaGetErrorString(err));
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        attr_set = true;
    }
    const int sw = C::W * 2;
    CUtensorMap tq = make_tensor_map_4d(q, HD, p.N, C::W, 128, sw);
    CUtensorMap tk = make_tensor_map_4d(k, HD, p.N, C::W, kNK, sw);
    CUtensorMap tv = make_tensor_map_4d(v, HD, p.N, C::W, kVT, sw);
    CUtensorMap to = make_tensor_map_4d(o, HD, p.N, 32, 128, 64);  // store box: 32 columns x 128 rows, SWIZZLE_64B
    const int grid = p.total < num_sms ? p.total : num_sms;
    kern<<<grid, kPThreads, C::kSmem, stream>>>(tq, tk, tv, to, p);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess)
        throw std::runtime_error(std::string("attention persist launch: ") + cudaGetErrorString(err));
}

// Instantiated for hd = 160 only: where two one-shot CTAs fit an SM (hd <= 128) those win.
bool attention_fwd_persist_supported(int N, int hd) { return N > 128 && N <= 256 && N % 2 == 0 && hd == 160; }

}  // namespace

// Optional in-kernel timeline (SURVEY 5.1): clock64 stamps of CTA 0's producer / MMA / softmax roles, 16 per work item.
static long long* g_trace = nullptr;
static int g_trace_items = 0;
void attention_set_trace(long long* buf, int items) { g_trace = buf, g_trace_items = items; }

void attention_fwd_persist(const __nv_bfloat16* qkv, int64_t ld_qkv, __nv_bfloat16* out, float* lse, int B, int N, int H,
                           int hd, cudaStream_t stream) {
    if (!attention_fwd_persist_supported(N, hd))
        throw std::runtime_error("attention_fwd_persist: unsupported (N, head_dim)");
    const int D = H * hd;
    const auto [q, k, v] = qkv_operands(qkv, ld_qkv, B, N, H, hd);
    PersistParams p;
    p.N = N, p.H = H, p.B = B, p.D = D;
    p.nq = (N + 127) / 128;
    p.nkt = (N + kVT - 1) / kVT;
    p.total = B * H * p.nq;
    p.scale = 1.0f / sqrtf(static_cast<float>(hd));
    p.scale_log2 = p.scale * 1.4426950408889634f;
    p.out = out, p.lse = lse;
    p.trace = g_trace, p.trace_items = g_trace_items;
    const GemmOperand o = head_operand(out, D, B, N, H, hd);  // what the epilogue's TMA stores address
    if (N % kVT != 0) launch_persist<160, true>(q, k, v, o, p, stream);  // key columns beyond N: ragged last tile
    else launch_persist<160, false>(q, k, v, o, p, stream);
}

}  // namespace b200
