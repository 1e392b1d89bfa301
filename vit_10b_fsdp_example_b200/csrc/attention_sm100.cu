// Fused multi-head attention forward for sm_100a: softmax(Q K^T * hd^-1/2) V for one (image, head, 128-query
// half) per CTA, for sequence lengths up to 256 tokens (ViT-10B: 256, ViT-L: 196).
//
//   TMA     : Q [128 x hd], K [NK x hd], V [NK x hd] are read *in place* from the packed qkv activation
//             ([tokens, 3*D], head h of q at columns h*hd) through 4-D tensor maps -- no permute / split copies.
//   tcgen05 : S = Q K^T (M=128, N=NK, fp32 accumulators in TMEM), then O = P V with P (bf16) staged in shared
//             memory *over the dead K tile* and V consumed as an MN-major operand (no transpose).
//             O re-uses the TMEM columns of S, so a CTA needs only NK columns and two CTAs fit an SM for hd=64.
//   softmax : one thread per query row straight out of TMEM (tcgen05.ld), exp2 with the scale folded in,
//             two passes (max, then exp/sum), un-normalised P to smem, 1/sum applied to O in the epilogue.
//   outputs : O [tokens, D] bf16, optionally the log-sum-exp per row (fp32) for the fused backward.
//
// Scores never reach HBM.  Replaces timm Attention's materialised [B,H,N,N] softmax
// (reference run_vit_training.py:134 -> timm Block -> Attention).
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>

#include "attention_sm100.h"
#include "gemm_sm100.h"
#include "ptx.cuh"

namespace b200 {

namespace {

constexpr int kAttnThreads = 192;  // warp0: TMA + MMA issue, warp1: TMEM alloc, warps 2-5: softmax / epilogue

struct AttnParams {
    int N;             // tokens per image
    int H, B;
    int D;             // H * hd
    float scale_log2;  // hd^-1/2 * log2(e)
    float scale;       // hd^-1/2
    __nv_bfloat16* out;  // [B*N, D]
    float* lse;          // [B*H, N] or null
};

template <int HD, int NK>
__global__ void __launch_bounds__(kAttnThreads) attn_fwd_sm100_kernel(const __grid_constant__ CUtensorMap tmap_q,
                                                                     const __grid_constant__ CUtensorMap tmap_k,
                                                                     const __grid_constant__ CUtensorMap tmap_v,
                                                                     const AttnParams p) {
    // hd-contiguous tiles use the widest swizzle atom that divides hd: 64 elements (SW128) or 32 (SW64)
    constexpr int W = (HD % 64 == 0) ? 64 : 32;
    constexpr int kAtoms = HD / W;
    constexpr uint32_t kLayout = (W == 64) ? 2u : 4u;
    constexpr int kRowBytes = W * 2;                 // bytes of one row inside an atom (128 or 64)
    constexpr int kQBytes = 128 * HD * 2;
    constexpr int kKBytes = NK * HD * 2;
    constexpr int kPBytes = 128 * NK * 2;
    constexpr int kKPBytes = kKBytes > kPBytes ? kKBytes : kPBytes;  // P is staged over the dead K tile
    static_assert(HD % 32 == 0 && HD <= 256 && HD <= NK, "unsupported head dim");
    static_assert(NK == 128 || NK == 256, "keys are padded to 128 or 256");

    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* sQ = smem;
    uint8_t* sK = sQ + kQBytes;       // also P
    uint8_t* sV = sK + kKPBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sV + kKBytes);
    uint64_t* bar_qk = bars;          // TMA Q + K landed
    uint64_t* bar_v = bars + 1;       // TMA V landed
    uint64_t* bar_s = bars + 2;       // S = Q K^T complete (tcgen05.commit)
    uint64_t* bar_p = bars + 3;       // P written by the 4 softmax warps
    uint64_t* bar_o = bars + 4;       // O = P V complete
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 5);

    const uint32_t warp_idx = threadIdx.x / 32;
    const uint32_t lane = lane_id();
    const int qhalf = blockIdx.x;  // which 128-query block
    const int h = blockIdx.y, b = blockIdx.z;

    if (warp_idx == 0 && elect_one()) {
        prefetch_tmap(&tmap_q);
        prefetch_tmap(&tmap_k);
        prefetch_tmap(&tmap_v);
        mbar_init(bar_qk, 1);
        mbar_init(bar_v, 1);
        mbar_init(bar_s, 1);
        mbar_init(bar_p, 4);
        mbar_init(bar_o, 1);
        fence_mbar_init();
    }
    if (warp_idx == 1) tmem_alloc<1>(tmem_ptr_smem, NK);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp_idx == 0) {
        if (elect_one()) {
            // ---- loads: one box per swizzle atom (W hd-columns x rows) ----
            mbar_arrive_expect_tx(bar_qk, kQBytes + kKBytes);
#pragma unroll
            for (int a = 0; a < kAtoms; ++a) {
                tma_load_4d(&tmap_q, bar_qk, sQ + a * (128 * kRowBytes), a * W, qhalf * 128, h, b);
                tma_load_4d(&tmap_k, bar_qk, sK + a * (NK * kRowBytes), a * W, 0, h, b);
            }
            mbar_arrive_expect_tx(bar_v, kKBytes);
#pragma unroll
            for (int a = 0; a < kAtoms; ++a) tma_load_4d(&tmap_v, bar_v, sV + a * (NK * kRowBytes), a * W, 0, h, b);

            // ---- S = Q K^T : A = Q (K-major), B = K (K-major), reduce over hd ----
            mbar_wait(bar_qk, 0);
            tc_fence_after();
            constexpr uint32_t idesc_s = make_idesc_bf16(128, NK, 0, 0);
            constexpr uint32_t kSbo = 8 * kRowBytes;
#pragma unroll
            for (int k = 0; k < HD / 16; ++k) {
                const int atom = (k * 16) / W, within = (k * 16) % W;
                const uint64_t da = make_smem_desc(smem_u32(sQ) + atom * (128 * kRowBytes) + within * 2, 0, kSbo, kLayout);
                const uint64_t db = make_smem_desc(smem_u32(sK) + atom * (NK * kRowBytes) + within * 2, 0, kSbo, kLayout);
                umma_bf16<1>(tmem_base, da, db, idesc_s, k > 0 ? 1u : 0u);
            }
            umma_commit<1>(bar_s);

            // ---- O = P V : A = P (K-major SW128 over the K tile), B = V (MN-major), reduce over keys ----
            mbar_wait(bar_p, 0);
            mbar_wait(bar_v, 0);
            tc_fence_after();
            constexpr uint32_t idesc_o = make_idesc_bf16(128, HD, 0, 1);
#pragma unroll
            for (int k = 0; k < NK / 16; ++k) {
                const int patom = (k * 16) / 64, pwithin = (k * 16) % 64;
                const uint64_t da = make_smem_desc(smem_u32(sK) + patom * (128 * 128) + pwithin * 2, 0, 1024, 2u);
                // MN-major: 8-key groups are 8*rowbytes apart (SBO), hd atoms are NK*rowbytes apart (LBO)
                const uint64_t db = make_smem_desc(smem_u32(sV) + k * 16 * kRowBytes, NK * kRowBytes, kSbo, kLayout);
                umma_bf16<1>(tmem_base, da, db, idesc_o, k > 0 ? 1u : 0u);
            }
            umma_commit<1>(bar_o);
        }
    } else if (warp_idx >= 2) {
        // ---- softmax + epilogue: thread <-> query row (TMEM lane quarter = warp_idx % 4) ----
        const uint32_t quarter = warp_idx & 3;
        const uint32_t r = quarter * 32 + lane;          // row inside the 128-query block
        const int q = qhalf * 128 + static_cast<int>(r);  // token index of this query
        const bool row_ok = q < p.N;
        const uint32_t taddr = tmem_base + ((quarter * 32) << 16);
        mbar_wait(bar_s, 0);
        tc_fence_after();
        float mx = -INFINITY;
#pragma unroll 1
        for (int c = 0; c < NK / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32b_x32(taddr + c * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (c * 32 + j < p.N) mx = fmaxf(mx, __uint_as_float(v[j]));
        }
        const float m_scaled = mx * p.scale_log2;
        float sum = 0.f;
        const uint32_t prow = smem_u32(sK) + r * 128;
#pragma unroll 1
        for (int c = 0; c < NK / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32b_x32(taddr + c * 32, v);
            tmem_ld_wait();
            float e[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                e[j] = (c * 32 + j < p.N) ? exp2f(fmaf(__uint_as_float(v[j]), p.scale_log2, -m_scaled)) : 0.f;
                sum += e[j];
            }
            // P tile: K-major SWIZZLE_128B, 64-key atoms of [128 rows x 128 B]
#pragma unroll
            for (int j8 = 0; j8 < 4; ++j8) {
                const int col = c * 32 + j8 * 8;
                const uint32_t atom = col >> 6, chunk = (col & 63) >> 3;
                const uint32_t addr = prow + atom * (128 * 128) + ((chunk ^ (r & 7)) << 4);
                st_shared_v4(addr, pack_bf16x2(e[j8 * 8], e[j8 * 8 + 1]), pack_bf16x2(e[j8 * 8 + 2], e[j8 * 8 + 3]),
                             pack_bf16x2(e[j8 * 8 + 4], e[j8 * 8 + 5]), pack_bf16x2(e[j8 * 8 + 6], e[j8 * 8 + 7]));
            }
        }
        const float inv = 1.0f / sum;
        tc_fence_before();
        fence_proxy_async_smem();  // generic-proxy P writes -> async-proxy (tensor core) reads
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_p);

        const int64_t bh = static_cast<int64_t>(b) * p.H + h;
        if (p.lse != nullptr && row_ok) p.lse[bh * p.N + q] = mx * p.scale + __logf(sum);

        // ---- epilogue: O / sum -> bf16 -> out[token, h*hd + :] ----
        mbar_wait(bar_o, 0);
        tc_fence_after();
        __nv_bfloat16* orow = p.out + (static_cast<int64_t>(b) * p.N + q) * p.D + h * HD;
#pragma unroll 1
        for (int c = 0; c < HD / 32; ++c) {
            uint32_t v[32];
            tmem_ld_32x32b_x32(taddr + c * 32, v);
            tmem_ld_wait();
            if (row_ok) {
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    uint4 o;
                    o.x = pack_bf16x2(__uint_as_float(v[j8 * 8]) * inv, __uint_as_float(v[j8 * 8 + 1]) * inv);
                    o.y = pack_bf16x2(__uint_as_float(v[j8 * 8 + 2]) * inv, __uint_as_float(v[j8 * 8 + 3]) * inv);
                    o.z = pack_bf16x2(__uint_as_float(v[j8 * 8 + 4]) * inv, __uint_as_float(v[j8 * 8 + 5]) * inv);
                    o.w = pack_bf16x2(__uint_as_float(v[j8 * 8 + 6]) * inv, __uint_as_float(v[j8 * 8 + 7]) * inv);
                    *reinterpret_cast<uint4*>(orow + c * 32 + j8 * 8) = o;
                }
            }
        }
        tc_fence_before();
    }
    __syncthreads();
    if (warp_idx == 1) tmem_dealloc<1>(tmem_base, NK);
}

template <int HD, int NK>
void launch_attn(const GemmOperand& q, const GemmOperand& k, const GemmOperand& v, const AttnParams& p,
                 cudaStream_t stream) {
    constexpr int W = (HD % 64 == 0) ? 64 : 32;
    constexpr int kQBytes = 128 * HD * 2, kKBytes = NK * HD * 2, kPBytes = 128 * NK * 2;
    constexpr int kSmem = kQBytes + (kKBytes > kPBytes ? kKBytes : kPBytes) + kKBytes + 64;
    static_assert(kSmem <= 232448, "shared memory budget exceeded");
    auto kern = attn_fwd_sm100_kernel<HD, NK>;
    static bool attr_set = false;
    if (!attr_set) {
        cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
        if (err != cudaSuccess) throw std::runtime_error(std::string("attention smem attr: ") + cudaGetErrorString(err));
        attr_set = true;
    }
    const int sw = W * 2;
    CUtensorMap tq = make_tensor_map_4d(q, HD, p.N, W, 128, sw);
    CUtensorMap tk = make_tensor_map_4d(k, HD, p.N, W, NK, sw);
    CUtensorMap tv = make_tensor_map_4d(v, HD, p.N, W, NK, sw);
    dim3 grid((p.N + 127) / 128, p.H, p.B);
    kern<<<grid, kAttnThreads, kSmem, stream>>>(tq, tk, tv, p);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) throw std::runtime_error(std::string("attention launch: ") + cudaGetErrorString(err));
}

bool attention_fwd_supported(int N, int hd) { return N <= 256 && (hd == 64 || hd == 128 || hd == 160) && N % 2 == 0; }

}  // namespace

void attention_fwd(const __nv_bfloat16* qkv, int64_t ld_qkv, __nv_bfloat16* out, float* lse, int B, int N, int H,
                   int hd, cudaStream_t stream) {
    if (!attention_fwd_supported(N, hd)) throw std::runtime_error("attention_fwd: unsupported (N, head_dim)");
    const auto [q, k, v] = qkv_operands(qkv, ld_qkv, B, N, H, hd);
    AttnParams p;
    p.N = N, p.H = H, p.B = B, p.D = H * hd;
    p.scale = 1.0f / sqrtf(static_cast<float>(hd));
    p.scale_log2 = p.scale * 1.4426950408889634f;
    p.out = out, p.lse = lse;
    const bool small = N <= 128;  // keys padded to 128 instead of 256 (needs hd <= 128: O re-uses S's TMEM columns)
    if (hd == 64) {
        if (small) launch_attn<64, 128>(q, k, v, p, stream);
        else launch_attn<64, 256>(q, k, v, p, stream);
    } else if (hd == 128) {
        if (small) launch_attn<128, 128>(q, k, v, p, stream);
        else launch_attn<128, 256>(q, k, v, p, stream);
    } else {
        launch_attn<160, 256>(q, k, v, p, stream);
    }
}

}  // namespace b200
