// Host API of the fused tcgen05 attention kernels (attention_sm100.cu, attention_bwd_sm100.cu,
// attention_persist_sm100.cu, attention_bwd_persist_sm100.cu).  Which kernel runs for a shape is decided by the
// caller (ops/attention_plan.py); every entry point throws on a shape its kernels cannot run.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>

#include "gemm_sm100.h"

namespace b200 {

// A [B*N, ld] activation whose H heads of hd columns sit side by side (head h at column h*hd), viewed as the
// [B][H][N rows x hd columns] operand the attention tensor maps address.
inline GemmOperand head_operand(const __nv_bfloat16* base, int64_t ld, int B, int N, int H, int hd) {
    GemmOperand o;
    o.ptr = base, o.ld = ld;
    o.nb_inner = H, o.stride_b_inner = hd;
    o.nb_outer = B, o.stride_b_outer = static_cast<int64_t>(N) * ld;
    return o;
}

// q, k and v read in place from the packed [B*N, 3*H*hd] qkv activation.
struct QkvOperands {
    GemmOperand q, k, v;
};
inline QkvOperands qkv_operands(const __nv_bfloat16* qkv, int64_t ld_qkv, int B, int N, int H, int hd) {
    const int64_t D = static_cast<int64_t>(H) * hd;
    return {head_operand(qkv, ld_qkv, B, N, H, hd), head_operand(qkv + D, ld_qkv, B, N, H, hd),
            head_operand(qkv + 2 * D, ld_qkv, B, N, H, hd)};
}

// One-shot forward, N <= 256 (attention_sm100.cu).  qkv: packed [B*N, 3*H*hd] (row stride ld_qkv).
// out: [B*N, H*hd].  lse: [B*H, N] fp32 or null.
void attention_fwd(const __nv_bfloat16* qkv, int64_t ld_qkv, __nv_bfloat16* out, float* lse, int B, int N, int H,
                   int hd, cudaStream_t stream);

// Long-sequence forward (any even N; two passes over 64-key tiles, attention_bwd_sm100.cu): out + row log-sum-exp.
void attention_fwd_long(const __nv_bfloat16* qkv, int64_t ld_qkv, __nv_bfloat16* out, float* lse, int B, int N, int H,
                        int hd, cudaStream_t stream);

// Persistent, software-pipelined forward for hd = 160, 128 < N <= 256 (attention_persist_sm100.cu): out, optional lse.
// debug: clock64 stamps of CTA 0 (16 int64 slots per work item) written by the persistent forward; nullptr = off
void attention_set_trace(long long* buf, int items);
// same for the persistent backward: 16 slots per global tile of CTA 0; role 0 = dK/dV kernel, 1 = dQ kernel
void attention_bwd_set_trace(long long* buf, int tiles, int role);
void attention_fwd_persist(const __nv_bfloat16* qkv, int64_t ld_qkv, __nv_bfloat16* out, float* lse, int B, int N, int H,
                           int hd, cudaStream_t stream);

// Fused backward (attention_bwd_sm100.cu).  dout / out: [B*N, H*hd] gradient and forward output of the attention core,
// lse: [B*H, N] from the forward, delta: [B*H, N] fp32 workspace (written here), dqkv: packed [B*N, 3*H*hd].
// persist = true runs the persistent 8-softmax-warp variant (attention_bwd_persist_sm100.cu, hd = 160, N % 4 == 0)
// instead of the one-shot kernels; delta then holds two [B*H, N] planes.
void attention_bwd(const __nv_bfloat16* qkv, int64_t ld_qkv, const __nv_bfloat16* dout, int64_t ld_do,
                   const __nv_bfloat16* out, int64_t ld_o, const float* lse, float* delta, __nv_bfloat16* dqkv,
                   int B, int N, int H, int hd, cudaStream_t stream, bool persist = false, float* colsum = nullptr);
// colsum (optional, persistent kernels only): zero-initialised fp32 [3 * D]; receives the column sums of dq | dk | dv
// (the qkv bias gradient) straight from the epilogue's staging tiles.
void attention_bwd_persist_core(const __nv_bfloat16* qkv, int64_t ld_qkv, const __nv_bfloat16* dout, int64_t ld_do,
                                const float* lse, const float* delta, __nv_bfloat16* dqkv, float* colsum, int B, int N,
                                int H, int hd, cudaStream_t stream);

}  // namespace b200
