// pybind11 / ATen bindings for the sm_100a kernels.  Compiled by g++ (no CUDA device code here), so the
// .cu files stay free of the heavy torch headers and rebuild in seconds.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <cmath>
#include <optional>
#include <vector>

#include "attention_sm100.h"
#include "comm.h"
#include "elementwise.h"
#include "gemm_sm100.h"

namespace {

using torch::Tensor;
using OptT = std::optional<Tensor>;

inline const __nv_bfloat16* bf16_ptr(const Tensor& t) {
    TORCH_CHECK(t.is_cuda(), "expected a CUDA tensor");
    TORCH_CHECK(t.scalar_type() == at::kBFloat16, "expected a bf16 tensor");
    return reinterpret_cast<const __nv_bfloat16*>(t.data_ptr());
}
inline __nv_bfloat16* bf16_mut(Tensor& t) { return const_cast<__nv_bfloat16*>(bf16_ptr(t)); }
inline float* f32_ptr(const Tensor& t) {
    TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kFloat, "expected a CUDA fp32 tensor");
    return reinterpret_cast<float*>(t.data_ptr());
}
inline cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

// batch = [] or [nb_inner, nb_outer, a_sbi, a_sbo, b_sbi, b_sbo, d_sbi, d_sbo] (strides in elements)
void gemm(Tensor a, int64_t lda, int64_t major_a, Tensor b, int64_t ldb, int64_t major_b, Tensor d, int64_t ldd,
          int64_t M, int64_t N, int64_t K, OptT bias, OptT residual, int64_t ld_res, int64_t res_row_mod, OptT aux_in,
          int64_t ld_aux, OptT aux_out, int64_t ld_aux_out, OptT colsum, int64_t colsum_bi_stride, int64_t act,
          std::vector<int64_t> batch, int64_t block_n, int64_t max_ctas, std::vector<int64_t> ag) {
    c10::cuda::CUDAGuard guard(a.device());
    b200::GemmOperand A, B, D, X;
    A.ptr = bf16_ptr(a), A.ld = lda;
    B.ptr = bf16_ptr(b), B.ld = ldb;
    D.ptr = bf16_ptr(d), D.ld = ldd;
    if (!batch.empty()) {
        TORCH_CHECK(batch.size() == 8, "batch spec must have 8 entries");
        A.nb_inner = B.nb_inner = D.nb_inner = batch[0];
        A.nb_outer = B.nb_outer = D.nb_outer = batch[1];
        A.stride_b_inner = batch[2], A.stride_b_outer = batch[3];
        B.stride_b_inner = batch[4], B.stride_b_outer = batch[5];
        D.stride_b_inner = batch[6], D.stride_b_outer = batch[7];
    }
    b200::GemmEpilogue e;
    if (bias.has_value()) e.bias = bf16_ptr(*bias);
    if (residual.has_value()) e.residual = bf16_ptr(*residual), e.ld_res = ld_res, e.res_row_mod = (int)res_row_mod;
    if (aux_in.has_value()) e.aux_in = bf16_ptr(*aux_in), e.ld_aux = ld_aux;
    if (colsum.has_value()) e.colsum = f32_ptr(*colsum), e.colsum_bi_stride = colsum_bi_stride;
    e.act = static_cast<int>(act);
    if (aux_out.has_value()) {
        X = D;
        X.ptr = bf16_ptr(*aux_out), X.ld = ld_aux_out;
        e.has_aux_out = 1;
    }
    // ag = [] or [world, rank, rows_per_slab, slab_bytes, dst_ptr, flags_ptr, peer_src_0, ..., peer_src_{W-1}]
    b200::GemmAgFuse fuse;
    if (!ag.empty()) {
        TORCH_CHECK(ag.size() >= 6 && (int64_t)ag.size() == 6 + ag[0] && ag[0] <= 16, "bad AG-fusion spec");
        fuse.world = (int)ag[0], fuse.rank = (int)ag[1], fuse.rows_per_slab = (int)ag[2], fuse.slab_bytes = ag[3];
        fuse.dst = reinterpret_cast<void*>(ag[4]);
        fuse.flags = reinterpret_cast<uint32_t*>(ag[5]);
        for (int64_t r = 0; r < ag[0]; ++r) fuse.peer_src[r] = static_cast<uint64_t>(ag[6 + r]);
    }
    b200::gemm_bf16(A, (int)major_a, B, (int)major_b, D, aux_out.has_value() ? &X : nullptr, (int)M, (int)N, (int)K, e,
                    (int)block_n, (int)max_ctas, cur_stream(), ag.empty() ? nullptr : &fuse);
}

void layernorm_fwd(Tensor x, Tensor gamma, Tensor beta, Tensor y, Tensor mean, Tensor rstd, double eps) {
    c10::cuda::CUDAGuard guard(x.device());
    const int D = (int)x.size(-1);
    const int rows = (int)(x.numel() / D);
    b200::layernorm_fwd(bf16_ptr(x), bf16_ptr(gamma), bf16_ptr(beta), bf16_mut(y), f32_ptr(mean), f32_ptr(rstd), rows,
                        D, (float)eps, cur_stream());
}

void layernorm_bwd(Tensor dy, Tensor x, Tensor gamma, Tensor mean, Tensor rstd, OptT dres, Tensor dx, Tensor dgamma,
                   Tensor dbeta, OptT dxsum) {
    c10::cuda::CUDAGuard guard(x.device());
    const int D = (int)x.size(-1);
    const int rows = (int)(x.numel() / D);
    b200::layernorm_bwd(bf16_ptr(dy), bf16_ptr(x), bf16_ptr(gamma), f32_ptr(mean), f32_ptr(rstd),
                        dres.has_value() ? bf16_ptr(*dres) : nullptr, bf16_mut(dx), f32_ptr(dgamma), f32_ptr(dbeta),
                        dxsum.has_value() ? f32_ptr(*dxsum) : nullptr, rows, D, cur_stream());
}

void softmax_fwd(Tensor s, int64_t rows, int64_t n, int64_t ld, double scale) {
    c10::cuda::CUDAGuard guard(s.device());
    b200::softmax_fwd(bf16_mut(s), rows, (int)n, ld, (float)scale, cur_stream());
}
void softmax_bwd(Tensor dp, Tensor p, int64_t rows, int64_t n, int64_t ld, double scale) {
    c10::cuda::CUDAGuard guard(p.device());
    b200::softmax_bwd(bf16_mut(dp), bf16_ptr(p), rows, (int)n, ld, (float)scale, cur_stream());
}

void attention_fwd(Tensor qkv, Tensor out, OptT lse, int64_t B, int64_t N, int64_t H, int64_t hd) {
    c10::cuda::CUDAGuard guard(qkv.device());
    TORCH_CHECK(qkv.dim() == 2 && qkv.stride(1) == 1 && out.is_contiguous(), "attention_fwd: bad layouts");
    b200::attention_fwd(bf16_ptr(qkv), qkv.stride(0), bf16_mut(out), lse.has_value() ? f32_ptr(*lse) : nullptr, (int)B,
                        (int)N, (int)H, (int)hd, cur_stream());
}

void attention_fwd_long(Tensor qkv, Tensor out, Tensor lse, int64_t B, int64_t N, int64_t H, int64_t hd) {
    c10::cuda::CUDAGuard guard(qkv.device());
    TORCH_CHECK(qkv.dim() == 2 && qkv.stride(1) == 1 && out.is_contiguous() && lse.is_contiguous() &&
                    lse.numel() == B * H * N,
                "attention_fwd_long: bad layouts");
    b200::attention_fwd_long(bf16_ptr(qkv), qkv.stride(0), bf16_mut(out), f32_ptr(lse), (int)B, (int)N, (int)H, (int)hd,
                             cur_stream());
}

void attention_set_trace(OptT buf) {
    if (!buf.has_value()) {
        b200::attention_set_trace(nullptr, 0);
        return;
    }
    TORCH_CHECK(buf->is_cuda() && buf->scalar_type() == at::kLong && buf->is_contiguous(), "trace: CUDA int64 tensor");
    b200::attention_set_trace(reinterpret_cast<long long*>(buf->data_ptr()), (int)(buf->numel() / 16));
}
void attention_bwd_set_trace(OptT buf, int64_t role) {
    if (!buf.has_value()) {
        b200::attention_bwd_set_trace(nullptr, 0, 0);
        return;
    }
    TORCH_CHECK(buf->is_cuda() && buf->scalar_type() == at::kLong && buf->is_contiguous(), "trace: CUDA int64 tensor");
    b200::attention_bwd_set_trace(reinterpret_cast<long long*>(buf->data_ptr()), (int)(buf->numel() / 16), (int)role);
}
void attention_fwd_persist(Tensor qkv, Tensor out, OptT lse, int64_t B, int64_t N, int64_t H, int64_t hd) {
    c10::cuda::CUDAGuard guard(qkv.device());
    TORCH_CHECK(qkv.dim() == 2 && qkv.stride(1) == 1 && out.is_contiguous(), "attention_fwd_persist: bad layouts");
    b200::attention_fwd_persist(bf16_ptr(qkv), qkv.stride(0), bf16_mut(out), lse.has_value() ? f32_ptr(*lse) : nullptr,
                                (int)B, (int)N, (int)H, (int)hd, cur_stream());
}

void attention_bwd(Tensor qkv, Tensor dout, Tensor out, Tensor lse, Tensor delta, Tensor dqkv, OptT colsum, int64_t B,
                   int64_t N, int64_t H, int64_t hd, bool persist) {
    c10::cuda::CUDAGuard guard(qkv.device());
    TORCH_CHECK(qkv.dim() == 2 && qkv.stride(1) == 1 && dout.stride(1) == 1 && out.stride(1) == 1 &&
                    dqkv.is_contiguous() && lse.is_contiguous() && delta.is_contiguous(),
                "attention_bwd: bad layouts");
    TORCH_CHECK(lse.numel() == B * H * N && delta.numel() == (persist ? 2 : 1) * B * H * N && dqkv.size(1) == 3 * H * hd,
                "attention_bwd: bad shapes (delta needs two [B*H, N] planes for the persistent kernels)");
    TORCH_CHECK(!persist || N % 4 == 0, "attention_bwd: persistent kernels need N % 4 == 0");
    b200::attention_bwd(bf16_ptr(qkv), qkv.stride(0), bf16_ptr(dout), dout.stride(0), bf16_ptr(out), out.stride(0),
                        f32_ptr(lse), f32_ptr(delta), bf16_mut(dqkv), (int)B, (int)N, (int)H, (int)hd, cur_stream(),
                        persist, colsum.has_value() ? f32_ptr(*colsum) : nullptr);
}

void cross_entropy(Tensor logits, Tensor target, OptT dlogits, Tensor loss, OptT correct) {
    c10::cuda::CUDAGuard guard(logits.device());
    TORCH_CHECK(target.scalar_type() == at::kLong && target.is_cuda(), "target must be a CUDA int64 tensor");
    const int B = (int)logits.size(0), C = (int)logits.size(1);
    b200::cross_entropy(bf16_ptr(logits), reinterpret_cast<const int64_t*>(target.data_ptr()),
                        dlogits.has_value() ? bf16_mut(*dlogits) : nullptr, f32_ptr(loss),
                        correct.has_value() ? reinterpret_cast<int*>(correct->data_ptr()) : nullptr, B, C,
                        cur_stream());
}

void im2col(Tensor img, Tensor cols, int64_t P) {
    c10::cuda::CUDAGuard guard(img.device());
    TORCH_CHECK(img.is_contiguous() && img.dim() == 4 && img.size(1) == 3, "images must be contiguous [B,3,S,S]");
    const bool is_bf16 = img.scalar_type() == at::kBFloat16;
    TORCH_CHECK(is_bf16 || img.scalar_type() == at::kFloat, "images must be fp32 or bf16");
    b200::im2col(img.data_ptr(), is_bf16, bf16_mut(cols), (int)img.size(0), (int)img.size(2), (int)P,
                 (int)cols.size(1), cur_stream());
}

void gelu_fwd(Tensor u, Tensor g) {
    c10::cuda::CUDAGuard guard(u.device());
    b200::gelu_fwd(bf16_ptr(u), bf16_mut(g), u.numel(), cur_stream());
}
void dropout(Tensor x, Tensor y, double p, int64_t key) {
    c10::cuda::CUDAGuard guard(x.device());
    TORCH_CHECK(x.is_contiguous() && y.is_contiguous() && x.numel() == y.numel(), "dropout: contiguous, same size");
    b200::dropout(bf16_ptr(x), bf16_mut(y), x.numel(), (float)p, (uint64_t)key, cur_stream());
}
void meanpool_fwd(Tensor xn, Tensor pooled, int64_t B, int64_t N) {
    c10::cuda::CUDAGuard guard(xn.device());
    TORCH_CHECK(xn.is_contiguous() && pooled.is_contiguous() && xn.numel() == pooled.numel() * N, "meanpool: bad shapes");
    b200::meanpool_fwd(bf16_ptr(xn), bf16_mut(pooled), (int)B, (int)N, (int)(pooled.numel() / B), cur_stream());
}
void meanpool_bwd(Tensor dpooled, Tensor dxn, int64_t B, int64_t N) {
    c10::cuda::CUDAGuard guard(dxn.device());
    TORCH_CHECK(dxn.is_contiguous() && dpooled.is_contiguous() && dxn.numel() == dpooled.numel() * N, "meanpool: bad shapes");
    b200::meanpool_bwd(bf16_ptr(dpooled), bf16_mut(dxn), (int)B, (int)N, (int)(dpooled.numel() / B), cur_stream());
}
void dgelu_mul(Tensor dg, Tensor u, Tensor du) {
    c10::cuda::CUDAGuard guard(u.device());
    b200::dgelu_mul(bf16_ptr(dg), bf16_ptr(u), bf16_mut(du), u.numel(), cur_stream());
}

void colsum(Tensor x, Tensor out) {
    c10::cuda::CUDAGuard guard(x.device());
    const int C = (int)x.size(-1);
    b200::colsum(bf16_ptr(x), f32_ptr(out), x.numel() / C, C, cur_stream());
}

void sumsq(Tensor x, Tensor out) {
    c10::cuda::CUDAGuard guard(x.device());
    const bool is_bf16 = x.scalar_type() == at::kBFloat16;
    TORCH_CHECK(is_bf16 || x.scalar_type() == at::kFloat, "sumsq: fp32 or bf16 only");
    b200::sumsq(x.data_ptr(), is_bf16, x.numel(), f32_ptr(out), cur_stream());
}

void adamw_split(Tensor hi, Tensor lo, Tensor m, Tensor v, Tensor grad, OptT clip_coef, double lr, double beta1,
                 double beta2, double eps, double wd, int64_t step, OptT hyper) {
    c10::cuda::CUDAGuard guard(hi.device());
    TORCH_CHECK(hi.scalar_type() == at::kBFloat16 && lo.scalar_type() == at::kShort, "hi: bf16, lo: int16");
    const bool gbf = grad.scalar_type() == at::kBFloat16;
    b200::adamw_split(reinterpret_cast<uint16_t*>(hi.data_ptr()), reinterpret_cast<int16_t*>(lo.data_ptr()),
                      f32_ptr(m), f32_ptr(v), grad.data_ptr(), gbf, hi.numel(),
                      clip_coef.has_value() ? f32_ptr(*clip_coef) : nullptr, (float)lr, (float)beta1, (float)beta2,
                      (float)eps, (float)wd, (int)step, cur_stream(), hyper.has_value() ? f32_ptr(*hyper) : nullptr);
}

void adamw_fp32(Tensor w, Tensor m, Tensor v, Tensor grad, OptT clip_coef, double lr, double beta1, double beta2,
                double eps, double wd, int64_t step) {
    c10::cuda::CUDAGuard guard(w.device());
    const bool gbf = grad.scalar_type() == at::kBFloat16;
    b200::adamw_fp32(f32_ptr(w), f32_ptr(m), f32_ptr(v), grad.data_ptr(), gbf, w.numel(),
                     clip_coef.has_value() ? f32_ptr(*clip_coef) : nullptr, (float)lr, (float)beta1, (float)beta2,
                     (float)eps, (float)wd, (int)step, cur_stream());
}

void split_fp32(Tensor w, Tensor hi, Tensor lo) {
    c10::cuda::CUDAGuard guard(w.device());
    b200::split_fp32(f32_ptr(w), reinterpret_cast<uint16_t*>(hi.data_ptr()), reinterpret_cast<int16_t*>(lo.data_ptr()),
                     w.numel(), cur_stream());
}
void merge_fp32(Tensor hi, Tensor lo, Tensor w) {
    c10::cuda::CUDAGuard guard(w.device());
    b200::merge_fp32(reinterpret_cast<const uint16_t*>(hi.data_ptr()), reinterpret_cast<const int16_t*>(lo.data_ptr()),
                     f32_ptr(w), w.numel(), cur_stream());
}
void clip_coef(Tensor sumsq_in, double max_norm, Tensor coef, OptT norm_out) {
    c10::cuda::CUDAGuard guard(coef.device());
    b200::clip_coef(f32_ptr(sumsq_in), (float)max_norm, f32_ptr(coef),
                    norm_out.has_value() ? f32_ptr(*norm_out) : nullptr, cur_stream());
}

// ---- NVLink / NVSwitch collectives over symmetric memory (raw device pointers from torch symm_mem) ----
inline const int64_t* seg_ptr(const Tensor& t) {
    TORCH_CHECK(t.is_cuda() && t.scalar_type() == at::kLong && t.is_contiguous(), "segment table: CUDA int64");
    return reinterpret_cast<const int64_t*>(t.data_ptr());
}
void p2p_all_gather(std::vector<int64_t> peer_ptrs, int64_t rank, Tensor out, Tensor seg_table, int64_t total_chunks,
                    int64_t max_ctas) {
    c10::cuda::CUDAGuard guard(out.device());
    b200::p2p_all_gather(peer_ptrs, (int)rank, out.data_ptr(), seg_ptr(seg_table), (int)seg_table.size(0),
                         total_chunks, (int)max_ctas, cur_stream());
}
// Copy-engine transport of the all-gather: one asynchronous device-to-device copy per (parameter group, source rank)
// straight from the peer's symmetric shard into its final place in the gathered buffer.  No SM, no shared memory, no
// registers are taken from the GEMM running next to it, and the DMA engines keep the NVLink pipe full where SM-issued
// peer loads do not (63 GB/s at W = 4 for the pull kernel, profiles/r2_n4.md).  Graph-capturable (memcpy nodes).
void ce_all_gather(std::vector<int64_t> src_ptrs, std::vector<int64_t> dst_ptrs, std::vector<int64_t> nbytes) {
    TORCH_CHECK(src_ptrs.size() == dst_ptrs.size() && src_ptrs.size() == nbytes.size(), "ce_all_gather: ragged lists");
    cudaStream_t stream = cur_stream();
    for (size_t i = 0; i < src_ptrs.size(); ++i) {
        cudaError_t err = cudaMemcpyAsync(reinterpret_cast<void*>(dst_ptrs[i]), reinterpret_cast<const void*>(src_ptrs[i]),
                                          static_cast<size_t>(nbytes[i]), cudaMemcpyDeviceToDevice, stream);
        TORCH_CHECK(err == cudaSuccess, "ce_all_gather: ", cudaGetErrorString(err));
    }
}
// adam = [] or (hi, lo, m, v tensors given separately) + hyper = [lr, beta1, beta2, eps, wd, step]
bool make_adam(const OptT& hi, const OptT& lo, const OptT& m, const OptT& v, const std::vector<double>& hyper,
               b200::AdamFuse& a) {
    if (!hi.has_value()) return false;
    TORCH_CHECK(lo.has_value() && m.has_value() && v.has_value() && hyper.size() == 6, "bad fused-AdamW arguments");
    TORCH_CHECK(hi->scalar_type() == at::kBFloat16 && lo->scalar_type() == at::kShort, "hi: bf16, lo: int16");
    a.hi = reinterpret_cast<uint16_t*>(hi->data_ptr());
    a.lo = reinterpret_cast<int16_t*>(lo->data_ptr());
    a.m = f32_ptr(*m);
    a.v = f32_ptr(*v);
    a.lr = (float)hyper[0], a.beta1 = (float)hyper[1], a.beta2 = (float)hyper[2], a.eps = (float)hyper[3];
    a.wd = (float)hyper[4];
    a.inv_bc1 = 1.f / (1.f - powf(a.beta1, (float)hyper[5]));
    a.inv_bc2 = 1.f / (1.f - powf(a.beta2, (float)hyper[5]));
    return true;
}
inline uint32_t* seq_ptr(const OptT& t) {
    if (!t.has_value()) return nullptr;
    TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kInt, "sequence counters: CUDA int32 tensor");
    return reinterpret_cast<uint32_t*>(t->data_ptr());
}
// sync = [] (caller brackets with barriers) or [rank, world, slot_ready, slot_done, counter_idx] + flag_ptrs, seq_dev, cta_ctr
bool make_sync(const std::vector<int64_t>& sync, const std::vector<int64_t>& flag_ptrs, const OptT& seq_dev,
               const OptT& cta_ctr, b200::CommSync& cs) {
    if (sync.empty()) return false;
    TORCH_CHECK(sync.size() == 5 && seq_dev.has_value() && cta_ctr.has_value(), "bad collective sync arguments");
    cs.flag_ptrs = flag_ptrs;
    cs.rank = (int)sync[0], cs.world = (int)sync[1], cs.slot_ready = (int)sync[2], cs.slot_done = (int)sync[3];
    cs.counter_idx = (int)sync[4];
    cs.seq_dev = seq_ptr(seq_dev);
    cs.cta_ctr = seq_ptr(cta_ctr);
    return true;
}
void reduce_scatter(std::vector<int64_t> peer_ptrs, int64_t mc_ptr, int64_t rank, int64_t world, Tensor out,
                    Tensor seg_table, int64_t total_chunks, bool in_is_bf16, double scale, OptT sumsq_out,
                    int64_t max_ctas, std::vector<int64_t> sync, std::vector<int64_t> flag_ptrs, OptT seq_dev,
                    OptT cta_ctr, OptT hi, OptT lo, OptT m, OptT v, std::vector<double> hyper) {
    c10::cuda::CUDAGuard guard(out.device());
    b200::AdamFuse a;
    const bool fused = make_adam(hi, lo, m, v, hyper, a);
    b200::CommSync cs;
    const bool synced = make_sync(sync, flag_ptrs, seq_dev, cta_ctr, cs);
    b200::reduce_scatter(peer_ptrs, mc_ptr, (int)rank, (int)world, f32_ptr(out), seg_ptr(seg_table),
                         (int)seg_table.size(0), total_chunks, in_is_bf16, (float)scale,
                         sumsq_out.has_value() ? f32_ptr(*sumsq_out) : nullptr, (int)max_ctas, cur_stream(),
                         synced ? &cs : nullptr, fused ? &a : nullptr);
}
void all_reduce_mean(std::vector<int64_t> peer_ptrs, int64_t mc_ptr, int64_t rank, int64_t world, Tensor buf,
                     int64_t max_ctas, std::vector<int64_t> sync, std::vector<int64_t> flag_ptrs, OptT seq_dev,
                     OptT cta_ctr) {
    c10::cuda::CUDAGuard guard(buf.device());
    TORCH_CHECK(buf.scalar_type() == at::kBFloat16 && buf.is_contiguous(), "all_reduce_mean: contiguous bf16 buffer");
    b200::CommSync cs;
    TORCH_CHECK(make_sync(sync, flag_ptrs, seq_dev, cta_ctr, cs), "all_reduce_mean needs the flag protocol");
    b200::all_reduce_mean_bf16(peer_ptrs, mc_ptr, (int)rank, (int)world, buf.numel() * 2, 1.0f / (float)world,
                               (int)max_ctas, cur_stream(), &cs);
}
void signal_barrier(std::vector<int64_t> flag_ptrs, int64_t rank, int64_t world, int64_t slot, int64_t seq,
                    OptT seq_dev) {
    b200::signal_barrier(flag_ptrs, (int)rank, (int)world, (int)slot, (uint32_t)seq, cur_stream(), seq_ptr(seq_dev));
}
void allreduce_scalars(std::vector<int64_t> flag_ptrs, std::vector<int64_t> scratch_ptrs, int64_t rank, int64_t world,
                       int64_t slot, int64_t seq, Tensor vals, int64_t op, OptT seq_dev, int64_t counter_idx) {
    c10::cuda::CUDAGuard guard(vals.device());
    b200::allreduce_scalars(flag_ptrs, scratch_ptrs, (int)rank, (int)world, (int)slot, (uint32_t)seq, f32_ptr(vals),
                            (int)vals.numel(), (int)op, cur_stream(), seq_ptr(seq_dev), (int)counter_idx);
}
int64_t ag_chunk_bytes() { return b200::ag_chunk_bytes(); }
int64_t rs_chunk_elems() { return b200::rs_chunk_elems(); }
int64_t rs_chunk_vecs() { return b200::rs_chunk_vecs(); }

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
    m.doc() = "vit_10b_fsdp_example_b200 native sm_100a kernels";
    m.def("gemm", &gemm);
    m.def("layernorm_fwd", &layernorm_fwd);
    m.def("layernorm_bwd", &layernorm_bwd);
    m.def("softmax_fwd", &softmax_fwd);
    m.def("softmax_bwd", &softmax_bwd);
    m.def("attention_fwd", &attention_fwd);
    m.def("attention_fwd_long", &attention_fwd_long);
    m.def("attention_fwd_persist", &attention_fwd_persist);
    m.def("attention_set_trace", &attention_set_trace);
    m.def("attention_bwd_set_trace", &attention_bwd_set_trace);
    m.def("attention_bwd", &attention_bwd);
    m.def("cross_entropy", &cross_entropy);
    m.def("im2col", &im2col);
    m.def("gelu_fwd", &gelu_fwd);
    m.def("dgelu_mul", &dgelu_mul);
    m.def("dropout", &dropout);
    m.def("meanpool_fwd", &meanpool_fwd);
    m.def("meanpool_bwd", &meanpool_bwd);
    m.def("colsum", &colsum);
    m.def("sumsq", &sumsq);
    m.def("adamw_split", &adamw_split);
    m.def("adamw_fp32", &adamw_fp32);
    m.def("split_fp32", &split_fp32);
    m.def("merge_fp32", &merge_fp32);
    m.def("clip_coef", &clip_coef);
    m.def("p2p_all_gather", &p2p_all_gather);
    m.def("ce_all_gather", &ce_all_gather);
    m.def("reduce_scatter", &reduce_scatter);
    m.def("all_reduce_mean", &all_reduce_mean);
    m.def("rs_chunk_vecs", &rs_chunk_vecs);
    m.def("signal_barrier", &signal_barrier);
    m.def("allreduce_scalars", &allreduce_scalars);
    m.def("ag_chunk_bytes", &ag_chunk_bytes);
    m.def("rs_chunk_elems", &rs_chunk_elems);
}
