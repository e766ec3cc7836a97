// Python bindings (pybind11 over torch::Tensor) for the sm_100a kernels.  Every function launches on the
// current PyTorch CUDA stream, so the ops compose with torch streams and CUDA-graph capture.
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include "comm.h"
#include "attention.h"
#include "gemm.h"
#include "kernels.h"

namespace rb {
extern long long g_launch_count;
}

namespace {

using torch::Tensor;
using OptTensor = c10::optional<Tensor>;

cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

void chk_bf16(const Tensor& t, const char* name) {
  TORCH_CHECK(t.is_cuda(), name, " must be a CUDA tensor");
  TORCH_CHECK(t.scalar_type() == at::kBFloat16, name, " must be bfloat16");
}
void chk_2d_rowmajor(const Tensor& t, const char* name) {
  TORCH_CHECK(t.dim() == 2 && t.stride(1) == 1, name, " must be 2-D with unit inner stride");
}
const uint32_t* u32ptr(const OptTensor& t) {
  if (!t.has_value()) return nullptr;
  TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kInt, "seed tensor must be a CUDA int32 tensor");
  return reinterpret_cast<const uint32_t*>(t->data_ptr<int32_t>());
}
const float* f32ptr(const OptTensor& t) {
  if (!t.has_value()) return nullptr;
  TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kFloat, "expected a CUDA float32 tensor");
  return t->data_ptr<float>();
}

rb::Operand operand(const Tensor& t, bool mn_major, const char* name) {
  chk_bf16(t, name);
  chk_2d_rowmajor(t, name);
  rb::Operand o;
  o.ptr = t.data_ptr();
  o.ld = t.stride(0);
  o.mn_major = mn_major;
  return o;
}

rb::Fp8Out fp8_out(const OptTensor& q8, const OptTensor& inv_scale, const OptTensor& amax, int64_t rows, int64_t cols) {
  rb::Fp8Out f;
  if (!q8.has_value()) return f;
  TORCH_CHECK(q8->is_cuda() && q8->element_size() == 1 && q8->dim() == 2 && q8->stride(1) == 1 && q8->size(0) == rows && q8->size(1) == cols,
              "fp8 output: one-byte [rows, cols] tensor");
  TORCH_CHECK(inv_scale.has_value() && amax.has_value(), "fp8 output needs inv_scale and amax");
  f.q = reinterpret_cast<uint8_t*>(q8->data_ptr()); f.ld = q8->stride(0);
  f.inv_scale = f32ptr(inv_scale); f.amax = const_cast<float*>(f32ptr(amax));
  return f;
}

// out[M,N] = alpha*(a1·b1ᵀ + a2·b2ᵀ) (+ residual) (+ out)
void gemm(const Tensor& a1, const Tensor& b1, Tensor& out, int64_t M, int64_t N, int64_t K1, const OptTensor& a2, const OptTensor& b2,
          int64_t K2, bool a1_mn, bool b1_mn, int64_t n_per_group, int64_t a1_group_kofs, int64_t a2_group_kofs,
          const OptTensor& residual, double alpha, bool accumulate, int64_t block_n, int64_t split_k, int64_t b1_group_kofs,
          bool b1_local_n, int64_t m_per_group, int64_t b1_mn_ofs_per_mgroup, const OptTensor& bias, int64_t cta_pair, int64_t fp8,
          const OptTensor& alpha_dev) {
  c10::cuda::CUDAGuard guard(out.device());
  rb::GemmDesc d;
  d.cta_pair = (int)cta_pair;
  if (fp8) {
    // E4M3 bytes (torch.uint8 / float8_e4m3fn storage), K-major; leading dimensions in bytes
    TORCH_CHECK(!a1_mn && !b1_mn, "fp8 operands must be K-major");
    for (const Tensor* t : {&a1, &b1}) {
      TORCH_CHECK(t->is_cuda() && t->element_size() == 1 && t->dim() == 2 && t->stride(1) == 1, "fp8 operands: 2-D one-byte CUDA tensors");
    }
    d.a1.ptr = a1.data_ptr(); d.a1.ld = a1.stride(0); d.a1.mn_major = false;
    d.b1.ptr = b1.data_ptr(); d.b1.ld = b1.stride(0); d.b1.mn_major = false;
    d.fp8 = true; d.fp8_a_e5m2 = fp8 == 2;
  } else {
    d.a1 = operand(a1, a1_mn, "a1");
    d.b1 = operand(b1, b1_mn, "b1");
  }
  if (alpha_dev.has_value()) d.alpha_dev = f32ptr(alpha_dev);
  d.M = (int)M; d.N = (int)N; d.K1 = (int)K1; d.K2 = (int)K2;
  if (K2 > 0) {
    TORCH_CHECK(a2.has_value() && b2.has_value(), "a2/b2 required when K2 > 0");
    d.a2 = operand(*a2, false, "a2");
    d.b2 = operand(*b2, false, "b2");
  }
  d.n_per_group = (int)n_per_group; d.a1_group_kofs = (int)a1_group_kofs; d.a2_group_kofs = (int)a2_group_kofs;
  TORCH_CHECK(out.is_cuda() && out.dim() == 2 && out.stride(1) == 1, "out must be 2-D row-major CUDA");
  TORCH_CHECK(out.scalar_type() == at::kBFloat16 || out.scalar_type() == at::kFloat, "out must be bf16 or fp32");
  TORCH_CHECK(out.size(0) >= M && out.size(1) >= N, "out too small");
  d.out = out.data_ptr(); d.ldc = out.stride(0); d.out_f32 = out.scalar_type() == at::kFloat;
  d.accumulate = accumulate; d.alpha = (float)alpha; d.block_n = (int)block_n; d.split_k = (int)split_k;
  d.b1_group_kofs = (int)b1_group_kofs; d.b1_local_n = b1_local_n; d.m_per_group = (int)m_per_group;
  d.b1_mn_ofs_per_mgroup = (int)b1_mn_ofs_per_mgroup;
  if (residual.has_value()) {
    chk_bf16(*residual, "residual");
    chk_2d_rowmajor(*residual, "residual");
    d.residual = residual->data_ptr(); d.ldr = residual->stride(0);
  }
  if (bias.has_value()) {
    chk_bf16(*bias, "bias");
    TORCH_CHECK(bias->is_contiguous() && bias->numel() >= N, "bias must be contiguous [N]");
    d.bias = bias->data_ptr();
  }
  rb::gemm_bf16(d, cur_stream());
}

void rmsnorm_fwd(const Tensor& x, const Tensor& w, Tensor& y, Tensor& rstd, double eps, const OptTensor& xd, const OptTensor& seed,
                 std::vector<int64_t> keys, double p, const OptTensor& q8, const OptTensor& q_inv_scale, const OptTensor& q_amax) {
  chk_bf16(x, "x"); chk_bf16(w, "w"); chk_bf16(y, "y");
  TORCH_CHECK(x.is_contiguous() && y.is_contiguous() && w.is_contiguous(), "rmsnorm: contiguous tensors required");
  const int H = (int)x.size(-1);
  const int M = (int)(x.numel() / H);
  c10::cuda::CUDAGuard guard(x.device());
  uint32_t k[4] = {0, 0, 0, 0};
  int G = 0;
  void* xdp = nullptr;
  if (xd.has_value()) {
    chk_bf16(*xd, "xd");
    TORCH_CHECK(xd->is_contiguous(), "xd must be contiguous");
    G = (int)keys.size();
    TORCH_CHECK(G >= 1 && G <= 4 && xd->numel() == (int64_t)M * G * H, "xd must be [M, G*H]");
    for (int i = 0; i < G; ++i) k[i] = (uint32_t)keys[i];
    xdp = xd->data_ptr();
  }
  const uint32_t thr = (uint32_t)llround(p * 65536.0);
  rb::rmsnorm_fwd(x.data_ptr(), w.data_ptr(), y.data_ptr(), rstd.data_ptr<float>(), M, H, (float)eps, xdp, G, u32ptr(seed), k, thr,
                  (float)(1.0 / (1.0 - p)), fp8_out(q8, q_inv_scale, q_amax, M, H), cur_stream());
}

void rmsnorm_bwd(const Tensor& dy, const Tensor& x, const Tensor& w, const Tensor& rstd, const OptTensor& dx_add, Tensor& dx, Tensor& dw,
                 const OptTensor& ws, const OptTensor& ticket) {
  chk_bf16(dy, "dy"); chk_bf16(x, "x"); chk_bf16(w, "w"); chk_bf16(dx, "dx");
  TORCH_CHECK(dw.scalar_type() == at::kFloat && dw.is_contiguous(), "dw must be fp32");
  TORCH_CHECK(dy.is_contiguous() && x.is_contiguous() && dx.is_contiguous(), "rmsnorm_bwd: contiguous tensors required");
  const int H = (int)x.size(-1);
  const int M = (int)(x.numel() / H);
  c10::cuda::CUDAGuard guard(x.device());
  const void* add = nullptr;
  if (dx_add.has_value()) { chk_bf16(*dx_add, "dx_add"); TORCH_CHECK(dx_add->is_contiguous()); add = dx_add->data_ptr(); }
  float* wsp = nullptr;
  unsigned int* tk = nullptr;
  if (ws.has_value() && ticket.has_value()) {
    TORCH_CHECK(ws->scalar_type() == at::kFloat && ws->numel() >= (int64_t)rb::rmsnorm_bwd_ws_blocks() * H, "rmsnorm workspace too small");
    TORCH_CHECK(ticket->scalar_type() == at::kInt && ticket->numel() >= 1, "ticket must be int32");
    wsp = ws->data_ptr<float>();
    tk = reinterpret_cast<unsigned int*>(ticket->data_ptr<int32_t>());
  }
  rb::rmsnorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), rstd.data_ptr<float>(), add, dx.data_ptr(), dw.data_ptr<float>(), M, H,
                  wsp, tk, cur_stream());
}

void dropout_expand(const Tensor& x, Tensor& xd, const OptTensor& seed, std::vector<int64_t> keys, double p, const OptTensor& q8,
                    const OptTensor& q_inv_scale, const OptTensor& q_amax) {
  chk_bf16(x, "x"); chk_bf16(xd, "xd");
  TORCH_CHECK(x.is_contiguous() && xd.is_contiguous());
  const int H = (int)x.size(-1);
  const int M = (int)(x.numel() / H);
  const int G = (int)keys.size();
  TORCH_CHECK(xd.numel() == (int64_t)M * G * H, "xd must be [M, G*H]");
  uint32_t k[4] = {0, 0, 0, 0};
  for (int i = 0; i < G && i < 4; ++i) k[i] = (uint32_t)keys[i];
  c10::cuda::CUDAGuard guard(x.device());
  rb::dropout_expand(x.data_ptr(), xd.data_ptr(), M, H, G, u32ptr(seed), k, (uint32_t)llround(p * 65536.0), (float)(1.0 / (1.0 - p)),
                     fp8_out(q8, q_inv_scale, q_amax, M, H), cur_stream());
}

void dropout_combine(const OptTensor& base, const Tensor& parts, Tensor& out, const OptTensor& seed, std::vector<int64_t> keys, double p) {
  // parts: either [G, M, H] contiguous, or [M, G*H] row-major (group g at column offset g*H)
  chk_bf16(parts, "parts"); chk_bf16(out, "out");
  TORCH_CHECK(out.dim() == 2 && out.is_contiguous(), "out must be contiguous [M, H]");
  const int M = (int)out.size(0), H = (int)out.size(1);
  const int G = (int)keys.size();
  long long part_stride, ld_parts;
  if (parts.dim() == 3) {
    TORCH_CHECK(parts.is_contiguous() && parts.size(0) == G && parts.size(1) == M && parts.size(2) == H, "parts must be [G, M, H]");
    part_stride = (long long)M * H; ld_parts = H;
  } else {
    TORCH_CHECK(parts.dim() == 2 && parts.stride(1) == 1 && parts.size(0) == M && parts.size(1) == (int64_t)G * H, "parts must be [M, G*H]");
    part_stride = H; ld_parts = parts.stride(0);
  }
  uint32_t k[4] = {0, 0, 0, 0};
  for (int i = 0; i < G && i < 4; ++i) k[i] = (uint32_t)keys[i];
  const void* bp = nullptr;
  if (base.has_value()) { chk_bf16(*base, "base"); TORCH_CHECK(base->is_contiguous() && base->numel() == out.numel()); bp = base->data_ptr(); }
  c10::cuda::CUDAGuard guard(out.device());
  rb::dropout_combine(bp, parts.data_ptr(), part_stride, ld_parts, out.data_ptr(), M, H, G, u32ptr(seed), k,
                      (uint32_t)llround(p * 65536.0), (float)(1.0 / (1.0 - p)), cur_stream());
}

void fp8_quantize_weight(const Tensor& w, Tensor& w8, Tensor& scratch, Tensor& scale, Tensor& inv_scale, const OptTensor& w8t) {
  chk_bf16(w, "w"); chk_2d_rowmajor(w, "w");
  TORCH_CHECK(w8.is_cuda() && w8.element_size() == 1 && w8.dim() == 2 && w8.stride(1) == 1 && w8.sizes() == w.sizes(), "w8: one-byte tensor shaped like w");
  void* tp = nullptr;
  long long tld = 0;
  if (w8t.has_value()) {
    TORCH_CHECK(w8t->is_cuda() && w8t->element_size() == 1 && w8t->dim() == 2 && w8t->stride(1) == 1 && w8t->size(0) == w.size(1) && w8t->size(1) == w.size(0),
                "w8t: one-byte tensor shaped like w transposed");
    tp = w8t->data_ptr(); tld = w8t->stride(0);
  }
  c10::cuda::CUDAGuard guard(w.device());
  rb::fp8_quantize_weight(w.data_ptr(), w.stride(0), w8.data_ptr(), w8.stride(0), tp, tld, (int)w.size(0), (int)w.size(1),
                          const_cast<float*>(f32ptr(scratch)), const_cast<float*>(f32ptr(scale)), const_cast<float*>(f32ptr(inv_scale)),
                          cur_stream());
}
void fp8_quantize_act(const Tensor& x, Tensor& x8, const Tensor& inv_scale, const OptTensor& amax_cur, bool e5m2) {
  chk_bf16(x, "x"); chk_2d_rowmajor(x, "x");
  TORCH_CHECK(x8.is_cuda() && x8.element_size() == 1 && x8.dim() == 2 && x8.stride(1) == 1 && x8.sizes() == x.sizes(), "x8: one-byte tensor shaped like x");
  c10::cuda::CUDAGuard guard(x.device());
  rb::fp8_quantize_act(x.data_ptr(), x.stride(0), x8.data_ptr(), x8.stride(0), (int)x.size(0), (int)x.size(1), f32ptr(inv_scale),
                       const_cast<float*>(f32ptr(amax_cur)), e5m2, cur_stream());
}
void fp8_prep(Tensor& state, const Tensor& w_scale, Tensor& inv_sx, Tensor& alpha_main, Tensor& alpha_inv, double margin, int64_t n_e4m3) {
  const int n = (int)w_scale.numel();
  TORCH_CHECK(state.numel() == 2 * n && inv_sx.numel() == n && alpha_main.numel() == n && alpha_inv.numel() == n, "fp8_prep: size mismatch");
  TORCH_CHECK(state.is_contiguous() && w_scale.is_contiguous() && inv_sx.is_contiguous() && alpha_main.is_contiguous() && alpha_inv.is_contiguous());
  c10::cuda::CUDAGuard guard(state.device());
  rb::fp8_prep(const_cast<float*>(f32ptr(state)), f32ptr(w_scale), const_cast<float*>(f32ptr(inv_sx)), const_cast<float*>(f32ptr(alpha_main)),
               const_cast<float*>(f32ptr(alpha_inv)), n, (float)margin, n_e4m3 < 0 ? n : (int)n_e4m3, cur_stream());
}

// out[M,N] = dy[M,Kb]·W[Kb,N] + Σ_g keep_g ⊙ (du_g·A_g)/(1-p)     (fused input gradient of a stacked LoRA group)
void lora_dx(const OptTensor& dy, const OptTensor& w, const Tensor& du, const Tensor& a, Tensor& out, const OptTensor& seed,
             std::vector<int64_t> keys, double p, const OptTensor& base) {
  chk_bf16(du, "du"); chk_bf16(a, "a"); chk_bf16(out, "out");
  chk_2d_rowmajor(du, "du"); chk_2d_rowmajor(a, "a"); chk_2d_rowmajor(out, "out");
  const int G = (int)keys.size();
  TORCH_CHECK(G >= 1 && G <= 3, "lora_dx: 1..3 groups");
  rb::LoraDxDesc d;
  d.M = (int)du.size(0); d.N = (int)a.size(1); d.groups = G;
  TORCH_CHECK(du.size(1) % G == 0, "du must be [M, G*r]");
  d.r = (int)(du.size(1) / G);
  TORCH_CHECK(a.size(0) == du.size(1), "a must be [G*r, N]");
  TORCH_CHECK(out.size(0) == d.M && out.size(1) == d.N, "out must be [M, N]");
  if (base.has_value()) {
    // two-kernel form: base = dy·W from the plain GEMM, this launch adds the masked low-rank terms
    chk_bf16(*base, "base"); chk_2d_rowmajor(*base, "base");
    TORCH_CHECK(base->size(0) == d.M && base->size(1) == d.N, "base must be [M, N]");
    d.base = base->data_ptr(); d.ld_base = base->stride(0); d.Kb = 0;
  } else {
    TORCH_CHECK(dy.has_value() && w.has_value(), "lora_dx: pass (dy, w) or base");
    chk_bf16(*dy, "dy"); chk_bf16(*w, "w"); chk_2d_rowmajor(*dy, "dy"); chk_2d_rowmajor(*w, "w");
    d.Kb = (int)dy->size(1);
    TORCH_CHECK(dy->size(0) == d.M && w->size(0) == d.Kb && w->size(1) == d.N, "dy must be [M, Kb], w [Kb, N]");
    d.dy = dy->data_ptr(); d.ld_dy = dy->stride(0);
    d.w = w->data_ptr(); d.ld_w = w->stride(0);
  }
  d.du = du.data_ptr(); d.ld_du = du.stride(0);
  d.a = a.data_ptr(); d.ld_a = a.stride(0);
  d.out = out.data_ptr(); d.ldc = out.stride(0);
  d.drop_threshold16 = (uint32_t)llround(p * 65536.0);
  d.inv_keep = (float)(1.0 / (1.0 - p));
  d.seed_ptr = u32ptr(seed);
  for (int i = 0; i < G; ++i) d.seed_key[i] = (uint32_t)keys[i];
  c10::cuda::CUDAGuard guard(out.device());
  rb::lora_dx(d, cur_stream());
}

// causal flash attention over the packed (post-RoPE) qkv buffer [B*T, 3*nh*hd]
void attention_fwd(const Tensor& qkv, Tensor& out, Tensor& lse, int64_t B, int64_t T, int64_t nh, int64_t hd, double scale) {
  chk_bf16(qkv, "qkv"); chk_bf16(out, "out"); chk_2d_rowmajor(qkv, "qkv"); chk_2d_rowmajor(out, "out");
  TORCH_CHECK(qkv.size(0) == B * T && qkv.size(1) == 3 * nh * hd, "qkv must be [B*T, 3*nh*hd]");
  TORCH_CHECK(out.size(0) == B * T && out.size(1) == nh * hd, "out must be [B*T, nh*hd]");
  TORCH_CHECK(lse.is_cuda() && lse.scalar_type() == at::kFloat && lse.is_contiguous() && lse.numel() == B * nh * T, "lse must be fp32 [B, nh, T]");
  rb::AttnDesc d;
  d.qkv = qkv.data_ptr(); d.ld_qkv = qkv.stride(0); d.out = out.data_ptr(); d.ld_out = out.stride(0); d.lse = lse.data_ptr<float>();
  d.B = (int)B; d.T = (int)T; d.nh = (int)nh; d.hd = (int)hd; d.scale = (float)scale;
  c10::cuda::CUDAGuard guard(qkv.device());
  rb::attention_fwd(d, cur_stream());
}
void attention_bwd(const Tensor& qkv, const Tensor& out, const Tensor& dout, const Tensor& lse, Tensor& delta, Tensor& dqkv, int64_t B,
                   int64_t T, int64_t nh, int64_t hd, double scale, const OptTensor& ds_workspace) {
  chk_bf16(qkv, "qkv"); chk_bf16(out, "out"); chk_bf16(dout, "dout"); chk_bf16(dqkv, "dqkv");
  chk_2d_rowmajor(qkv, "qkv"); chk_2d_rowmajor(out, "out"); chk_2d_rowmajor(dout, "dout"); chk_2d_rowmajor(dqkv, "dqkv");
  TORCH_CHECK(qkv.size(0) == B * T && qkv.size(1) == 3 * nh * hd && dqkv.size(0) == B * T && dqkv.size(1) == 3 * nh * hd, "qkv / dqkv must be [B*T, 3*nh*hd]");
  TORCH_CHECK(out.size(0) == B * T && out.size(1) == nh * hd && dout.size(0) == B * T && dout.size(1) == nh * hd, "out / dout must be [B*T, nh*hd]");
  TORCH_CHECK(lse.scalar_type() == at::kFloat && lse.is_contiguous() && lse.numel() == B * nh * T, "lse must be fp32 [B, nh, T]");
  TORCH_CHECK(delta.is_cuda() && delta.scalar_type() == at::kFloat && delta.is_contiguous() && delta.numel() == B * nh * T, "delta must be fp32 [B, nh, T]");
  rb::AttnBwdDesc d;
  d.qkv = qkv.data_ptr(); d.ld_qkv = qkv.stride(0); d.out = out.data_ptr(); d.ld_out = out.stride(0);
  d.dout = dout.data_ptr(); d.ld_dout = dout.stride(0); d.lse = lse.data_ptr<float>(); d.delta = delta.data_ptr<float>();
  d.dqkv = dqkv.data_ptr(); d.ld_dqkv = dqkv.stride(0);
  d.B = (int)B; d.T = (int)T; d.nh = (int)nh; d.hd = (int)hd; d.scale = (float)scale;
  if (ds_workspace.has_value()) {
    chk_bf16(*ds_workspace, "ds_workspace");
    TORCH_CHECK(ds_workspace->is_contiguous() && ds_workspace->numel() >= rb::attention_ds_workspace_elems((int)B, (int)T, (int)nh),
                "ds_workspace too small (attention_ds_workspace_elems)");
    d.ds_workspace = ds_workspace->data_ptr();
  }
  c10::cuda::CUDAGuard guard(qkv.device());
  rb::attention_bwd(d, cur_stream());
}

// bf16 cos / sin tables [n_pos, rotary_dim] covering positions pos0 .. pos0 + T - 1 (the kernels read them unchecked)
void chk_rope_tables(const Tensor& cos, const Tensor& sin, int64_t T, int64_t pos0, int64_t rotary_dim, int64_t hd) {
  chk_bf16(cos, "cos"); chk_bf16(sin, "sin");
  TORCH_CHECK(cos.dim() == 2 && cos.is_contiguous() && sin.is_contiguous() && cos.size(1) == rotary_dim && sin.sizes() == cos.sizes(),
              "cos/sin must be contiguous [n_pos, rotary_dim]");
  TORCH_CHECK(rotary_dim > 0 && rotary_dim <= hd, "rotary_dim must be in (0, head_dim]");
  TORCH_CHECK(pos0 >= 0 && T + pos0 <= cos.size(0), "rotary table too short");
}

void rope_inplace(Tensor& buf, int64_t T, int64_t n_rot_heads, int64_t hd, int64_t rotary_dim, const Tensor& cos, const Tensor& sin,
                  bool backward, int64_t pos0) {
  chk_bf16(buf, "buf");
  chk_2d_rowmajor(buf, "buf");
  chk_rope_tables(cos, sin, T, pos0, rotary_dim, hd);
  c10::cuda::CUDAGuard guard(buf.device());
  rb::rope_inplace(buf.data_ptr(), buf.stride(0), (int)buf.size(0), (int)T, (int)n_rot_heads, (int)hd, (int)rotary_dim, cos.data_ptr(),
                   sin.data_ptr(), backward, (int)pos0, cur_stream());
}

void rope_pack_bwd(const Tensor& dq, const Tensor& dk, const Tensor& dv, Tensor& out, int64_t rotary_dim, const Tensor& cos,
                   const Tensor& sin, int64_t pos0) {
  chk_bf16(dq, "dq"); chk_bf16(dk, "dk"); chk_bf16(dv, "dv"); chk_bf16(out, "out"); chk_2d_rowmajor(out, "out");
  TORCH_CHECK(dq.dim() == 4 && dq.stride(3) == 1 && dq.sizes() == dk.sizes() && dq.sizes() == dv.sizes(), "dq/dk/dv must be [B, nh, T, hd]");
  TORCH_CHECK(dq.strides() == dk.strides() && dq.strides() == dv.strides(), "dq/dk/dv must share strides");
  const int B = (int)dq.size(0), nh = (int)dq.size(1), T = (int)dq.size(2), hd = (int)dq.size(3);
  TORCH_CHECK(out.size(0) == (int64_t)B * T && out.size(1) == 3 * (int64_t)nh * hd, "out must be [B*T, 3*nh*hd]");
  chk_rope_tables(cos, sin, T, pos0, rotary_dim, hd);
  for (const Tensor* t : {&dq, &dk, &dv}) TORCH_CHECK((reinterpret_cast<uintptr_t>(t->data_ptr()) & 15) == 0, "16-byte alignment required");
  c10::cuda::CUDAGuard guard(out.device());
  rb::rope_pack_bwd(dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), dq.stride(0), dq.stride(1), dq.stride(2), out.data_ptr(), out.stride(0), B, T, nh,
                    hd, (int)rotary_dim, cos.data_ptr(), sin.data_ptr(), (int)pos0, cur_stream());
}

void swiglu_fwd(const Tensor& gu, Tensor& h, const OptTensor& hd, const OptTensor& seed, int64_t key, double p, const OptTensor& q8,
                const OptTensor& q_inv_scale, const OptTensor& q_amax) {
  chk_bf16(gu, "gu"); chk_bf16(h, "h"); chk_2d_rowmajor(gu, "gu"); chk_2d_rowmajor(h, "h");
  const int F = (int)h.size(1);
  TORCH_CHECK(gu.size(1) == 2 * F && gu.size(0) == h.size(0));
  void* hdp = nullptr;
  long long ldhd = 0;
  if (hd.has_value()) {
    chk_bf16(*hd, "hd"); chk_2d_rowmajor(*hd, "hd");
    TORCH_CHECK(hd->size(0) == h.size(0) && hd->size(1) == F, "hd must be [M, F]");
    hdp = hd->data_ptr(); ldhd = hd->stride(0);
  }
  c10::cuda::CUDAGuard guard(gu.device());
  rb::swiglu_fwd(gu.data_ptr(), gu.stride(0), h.data_ptr(), h.stride(0), (int)h.size(0), F, hdp, ldhd, u32ptr(seed), (uint32_t)key,
                 (uint32_t)llround(p * 65536.0), (float)(1.0 / (1.0 - p)), fp8_out(q8, q_inv_scale, q_amax, h.size(0), F), cur_stream());
}
void swiglu_bwd(const Tensor& dh, const Tensor& gu, Tensor& dgu) {
  chk_bf16(dh, "dh"); chk_bf16(gu, "gu"); chk_bf16(dgu, "dgu");
  chk_2d_rowmajor(dh, "dh"); chk_2d_rowmajor(gu, "gu"); chk_2d_rowmajor(dgu, "dgu");
  const int F = (int)dh.size(1);
  TORCH_CHECK(gu.size(1) == 2 * F && dgu.size(1) == 2 * F);
  c10::cuda::CUDAGuard guard(gu.device());
  rb::swiglu_bwd(dh.data_ptr(), dh.stride(0), gu.data_ptr(), gu.stride(0), dgu.data_ptr(), dgu.stride(0), (int)dh.size(0), F, cur_stream());
}

// ---------------------------------------------------------------------------------------------- block-scaled MXFP8
int64_t mx_sf_bytes(int64_t rows, int64_t k) { return rb::mx_sf_bytes(rows, k); }
void mx_quantize_rows(const Tensor& x, Tensor& q, Tensor& sf) {
  chk_bf16(x, "x"); chk_2d_rowmajor(x, "x");
  TORCH_CHECK(q.is_cuda() && q.scalar_type() == at::kByte && q.dim() == 2 && q.stride(1) == 1 && q.size(0) >= x.size(0), "q must be uint8 [M, Kpad]");
  TORCH_CHECK(sf.is_cuda() && sf.scalar_type() == at::kByte && sf.is_contiguous() && sf.numel() >= rb::mx_sf_bytes(x.size(0), x.size(1)), "sf too small");
  c10::cuda::CUDAGuard guard(x.device());
  rb::mx_quantize_rows(x.data_ptr(), x.stride(0), q.data_ptr(), q.stride(0), sf.data_ptr(), (int)x.size(0), (int)x.size(1), cur_stream());
}
void mx_quantize_weight_2d(const OptTensor& w, const OptTensor& delta, Tensor& q, Tensor& sf_fwd, Tensor& sf_bwd, int64_t N, int64_t K) {
  TORCH_CHECK(q.is_cuda() && q.scalar_type() == at::kByte && q.dim() == 2 && q.stride(1) == 1, "q must be uint8 [Npad, Kpad]");
  TORCH_CHECK(q.size(0) >= (N + 127) / 128 * 128 && q.size(1) >= (K + 127) / 128 * 128, "q must be padded to multiples of 128 in both dimensions");
  TORCH_CHECK(sf_fwd.scalar_type() == at::kByte && sf_bwd.scalar_type() == at::kByte && sf_fwd.is_contiguous() && sf_bwd.is_contiguous());
  TORCH_CHECK(sf_fwd.numel() >= rb::mx_sf_bytes(N, K) && sf_bwd.numel() >= rb::mx_sf_bytes(K, N), "scale buffers too small");
  const void* wp = nullptr; long long ldw = 0;
  if (w.has_value()) { chk_bf16(*w, "w"); chk_2d_rowmajor(*w, "w"); TORCH_CHECK(w->size(0) == N && w->size(1) == K); wp = w->data_ptr(); ldw = w->stride(0); }
  const float* dp = nullptr; long long ldd = 0;
  if (delta.has_value()) {
    TORCH_CHECK(delta->scalar_type() == at::kFloat && delta->dim() == 2 && delta->stride(1) == 1 && delta->size(0) == N && delta->size(1) == K);
    dp = delta->data_ptr<float>(); ldd = delta->stride(0);
  }
  c10::cuda::CUDAGuard guard(q.device());
  rb::mx_quantize_weight_2d(wp, ldw, q.data_ptr(), sf_fwd.data_ptr(), dp, ldd, q.data_ptr(), q.stride(0), sf_fwd.data_ptr(), sf_bwd.data_ptr(),
                            (int)N, (int)K, cur_stream());
}
void mx_dequantize_weight(const Tensor& q, const Tensor& sf_fwd, Tensor& out) {
  chk_bf16(out, "out"); chk_2d_rowmajor(out, "out");
  TORCH_CHECK(q.scalar_type() == at::kByte && q.dim() == 2 && q.stride(1) == 1 && sf_fwd.scalar_type() == at::kByte);
  c10::cuda::CUDAGuard guard(q.device());
  rb::mx_dequantize_weight(q.data_ptr(), q.stride(0), sf_fwd.data_ptr(), out.data_ptr(), out.stride(0), (int)out.size(0), (int)out.size(1), cur_stream());
}
void gemm_mx(const Tensor& a, const Tensor& sfa, const Tensor& b, const Tensor& sfb, Tensor& out, int64_t M, int64_t N, int64_t K, bool b_mn_major,
             const OptTensor& a2, const OptTensor& b2, const OptTensor& residual) {
  TORCH_CHECK(a.is_cuda() && a.scalar_type() == at::kByte && b.scalar_type() == at::kByte && a.dim() == 2 && b.dim() == 2 && a.stride(1) == 1 && b.stride(1) == 1);
  TORCH_CHECK(sfa.scalar_type() == at::kByte && sfb.scalar_type() == at::kByte && sfa.is_contiguous() && sfb.is_contiguous());
  chk_bf16(out, "out"); chk_2d_rowmajor(out, "out");
  const int64_t Kpad = (K + 127) / 128 * 128;
  TORCH_CHECK(a.size(0) >= M && a.size(1) >= Kpad, "a must be [>= M, >= Kpad] fp8 bytes");
  if (b_mn_major) {
    TORCH_CHECK(b.size(0) >= Kpad && b.size(1) >= N, "MN-major b must be [>= Kpad rows, >= N]");
  } else {
    TORCH_CHECK(b.size(0) >= N && b.size(1) >= Kpad, "K-major b must be [>= N, >= Kpad]");
  }
  TORCH_CHECK(sfa.numel() >= rb::mx_sf_bytes(M, K) && sfb.numel() >= rb::mx_sf_bytes(N, K), "scale buffers too small");
  TORCH_CHECK(out.size(0) == M && out.size(1) == N);
  rb::MxGemmDesc d;
  d.a = a.data_ptr(); d.lda = a.stride(0); d.b = b.data_ptr(); d.ldb = b.stride(0); d.sfa = sfa.data_ptr(); d.sfb = sfb.data_ptr();
  d.b_mn_major = b_mn_major; d.M = (int)M; d.N = (int)N; d.K = (int)K; d.out = out.data_ptr(); d.ldc = out.stride(0);
  if (a2.has_value()) {
    TORCH_CHECK(b2.has_value(), "a2 needs b2");
    chk_bf16(*a2, "a2"); chk_bf16(*b2, "b2"); chk_2d_rowmajor(*a2, "a2"); chk_2d_rowmajor(*b2, "b2");
    TORCH_CHECK(a2->size(0) == M && b2->size(0) == N && a2->size(1) == b2->size(1));
    d.a2 = a2->data_ptr(); d.lda2 = a2->stride(0); d.b2 = b2->data_ptr(); d.ldb2 = b2->stride(0); d.K2 = (int)a2->size(1);
  }
  if (residual.has_value()) {
    chk_bf16(*residual, "residual"); chk_2d_rowmajor(*residual, "residual");
    TORCH_CHECK(residual->size(0) == M && residual->size(1) == N);
    d.residual = residual->data_ptr(); d.ldr = residual->stride(0);
  }
  c10::cuda::CUDAGuard guard(a.device());
  rb::gemm_mx(d, cur_stream());
}

// ---------------------------------------------------------------------------------------------- GPT-NeoX / Pythia block
void layernorm_fwd(const Tensor& x, const Tensor& w, const OptTensor& b, Tensor& y, Tensor& mean, Tensor& rstd, double eps) {
  chk_bf16(x, "x"); chk_bf16(w, "weight"); chk_bf16(y, "y");
  TORCH_CHECK(x.is_contiguous() && y.is_contiguous() && w.is_contiguous() && x.dim() == 2 && w.numel() == x.size(1));
  TORCH_CHECK(mean.scalar_type() == at::kFloat && rstd.scalar_type() == at::kFloat && mean.numel() == x.size(0) && rstd.numel() == x.size(0));
  if (b.has_value()) { chk_bf16(*b, "bias"); TORCH_CHECK(b->is_contiguous() && b->numel() == x.size(1)); }
  c10::cuda::CUDAGuard guard(x.device());
  const bool ok = rb::layernorm_fwd(x.data_ptr(), w.data_ptr(), b.has_value() ? b->data_ptr() : nullptr, y.data_ptr(), mean.data_ptr<float>(),
                                    rstd.data_ptr<float>(), (int)x.size(0), (int)x.size(1), (float)eps, cur_stream());
  TORCH_CHECK(ok, "layernorm_fwd: hidden size must be a multiple of 8 and <= 4096");
}
void layernorm_bwd(const Tensor& dy, const Tensor& x, const Tensor& w, const Tensor& mean, const Tensor& rstd, Tensor& dx, Tensor& dw,
                   const OptTensor& db) {
  chk_bf16(dy, "dy"); chk_bf16(x, "x"); chk_bf16(w, "weight"); chk_bf16(dx, "dx");
  TORCH_CHECK(dy.is_contiguous() && x.is_contiguous() && dx.is_contiguous() && w.is_contiguous() && x.dim() == 2);
  TORCH_CHECK(dw.scalar_type() == at::kFloat && dw.is_contiguous() && dw.numel() == x.size(1));
  if (db.has_value()) TORCH_CHECK(db->scalar_type() == at::kFloat && db->is_contiguous() && db->numel() == x.size(1));
  c10::cuda::CUDAGuard guard(x.device());
  const bool ok = rb::layernorm_bwd(dy.data_ptr(), x.data_ptr(), w.data_ptr(), mean.data_ptr<float>(), rstd.data_ptr<float>(), dx.data_ptr(),
                                    dw.data_ptr<float>(), db.has_value() ? db->data_ptr<float>() : nullptr, (int)x.size(0), (int)x.size(1),
                                    cur_stream());
  TORCH_CHECK(ok, "layernorm_bwd: hidden size must be a multiple of 8 and <= 2048");
}
void gelu_fwd(const Tensor& z, Tensor& a, bool tanh_approx) {
  chk_bf16(z, "z"); chk_bf16(a, "a");
  TORCH_CHECK(z.is_contiguous() && a.is_contiguous() && z.numel() == a.numel());
  c10::cuda::CUDAGuard guard(z.device());
  rb::gelu_fwd(z.data_ptr(), a.data_ptr(), z.numel(), tanh_approx, cur_stream());
}
void gelu_bwd(const Tensor& da, const Tensor& z, Tensor& dz, bool tanh_approx) {
  chk_bf16(da, "da"); chk_bf16(z, "z"); chk_bf16(dz, "dz");
  TORCH_CHECK(da.is_contiguous() && z.is_contiguous() && dz.is_contiguous() && z.numel() == da.numel() && z.numel() == dz.numel());
  c10::cuda::CUDAGuard guard(z.device());
  rb::gelu_bwd(da.data_ptr(), z.data_ptr(), dz.data_ptr(), z.numel(), tanh_approx, cur_stream());
}
void neox_rope(Tensor& qkv, int64_t T, int64_t nh, int64_t hd, int64_t rot, const Tensor& cos, const Tensor& sin, int64_t pos0, bool inverse) {
  chk_bf16(qkv, "qkv"); chk_2d_rowmajor(qkv, "qkv");
  TORCH_CHECK(qkv.size(1) == nh * 3 * hd, "qkv must be [rows, nh * 3 * hd]");
  TORCH_CHECK(cos.scalar_type() == at::kFloat && sin.scalar_type() == at::kFloat && cos.is_contiguous() && sin.is_contiguous() &&
              cos.dim() == 2 && cos.size(1) == rot && sin.sizes() == cos.sizes() && T + pos0 <= cos.size(0), "cos / sin must be fp32 [n_pos, rot]");
  c10::cuda::CUDAGuard guard(qkv.device());
  rb::neox_rope(qkv.data_ptr(), qkv.stride(0), qkv.size(0), (int)T, (int)nh, (int)hd, (int)rot, cos.data_ptr<float>(), sin.data_ptr<float>(),
                (int)pos0, inverse, cur_stream());
}

void embedding_fwd(const Tensor& ids, const Tensor& table, Tensor& out) {
  chk_bf16(table, "table"); chk_bf16(out, "out");
  TORCH_CHECK(ids.is_cuda() && ids.scalar_type() == at::kLong && ids.is_contiguous() && table.is_contiguous() && out.is_contiguous());
  c10::cuda::CUDAGuard guard(out.device());
  rb::embedding_fwd(ids.data_ptr<int64_t>(), table.data_ptr(), out.data_ptr(), (int)ids.numel(), (int)table.size(1), cur_stream());
}
void embedding_bwd(const Tensor& ids, const Tensor& dout, Tensor& dtable, int64_t padding_idx) {
  chk_bf16(dout, "dout");
  TORCH_CHECK(dtable.scalar_type() == at::kFloat && dtable.is_contiguous() && dout.is_contiguous() && ids.is_contiguous());
  c10::cuda::CUDAGuard guard(dout.device());
  rb::embedding_bwd(ids.data_ptr<int64_t>(), dout.data_ptr(), dtable.data_ptr<float>(), (int)ids.numel(), (int)dtable.size(1), padding_idx,
                    cur_stream());
}

void embedding_bwd_sorted(const Tensor& sorted_ids, const Tensor& perm, const Tensor& dout, Tensor& dtable, int64_t padding_idx) {
  chk_bf16(dout, "dout");
  TORCH_CHECK(dtable.scalar_type() == at::kFloat && dtable.is_contiguous() && dout.is_contiguous());
  TORCH_CHECK(sorted_ids.scalar_type() == at::kLong && perm.scalar_type() == at::kLong && sorted_ids.is_contiguous() && perm.is_contiguous() &&
              sorted_ids.numel() == perm.numel());
  c10::cuda::CUDAGuard guard(dout.device());
  rb::embedding_bwd_sorted(sorted_ids.data_ptr<int64_t>(), perm.data_ptr<int64_t>(), dout.data_ptr(), dtable.data_ptr<float>(),
                           (int)sorted_ids.numel(), (int)dtable.size(1), padding_idx, cur_stream());
}

void cross_entropy_fwd_bwd(Tensor& logits, const Tensor& labels, int64_t V, double grad_scale, int64_t ignore_index, Tensor& loss_sum,
                           Tensor& count) {
  chk_bf16(logits, "logits"); chk_2d_rowmajor(logits, "logits");
  TORCH_CHECK(labels.is_cuda() && labels.scalar_type() == at::kLong && labels.is_contiguous() && labels.numel() == logits.size(0));
  TORCH_CHECK(loss_sum.scalar_type() == at::kFloat && count.scalar_type() == at::kFloat);
  c10::cuda::CUDAGuard guard(logits.device());
  rb::cross_entropy_fwd_bwd(logits.data_ptr(), logits.stride(0), labels.data_ptr<int64_t>(), (int)logits.size(0), (int)V, (float)grad_scale,
                            ignore_index, loss_sum.data_ptr<float>(), count.data_ptr<float>(), cur_stream());
}

void transpose(const Tensor& in, Tensor& out) {
  chk_bf16(in, "in"); chk_bf16(out, "out"); chk_2d_rowmajor(in, "in"); chk_2d_rowmajor(out, "out");
  TORCH_CHECK(out.size(0) == in.size(1) && out.size(1) == in.size(0));
  c10::cuda::CUDAGuard guard(in.device());
  rb::transpose_bf16(in.data_ptr(), in.stride(0), out.data_ptr(), out.stride(0), (int)in.size(0), (int)in.size(1), cur_stream());
}
void add(const Tensor& a, const Tensor& b, Tensor& out) {
  chk_bf16(a, "a"); chk_bf16(b, "b"); chk_bf16(out, "out");
  TORCH_CHECK(a.is_contiguous() && b.is_contiguous() && out.is_contiguous() && a.numel() == b.numel() && a.numel() == out.numel());
  c10::cuda::CUDAGuard guard(a.device());
  rb::add_bf16(a.data_ptr(), b.data_ptr(), out.data_ptr(), a.numel(), cur_stream());
}
void cast_f32_to_bf16(const Tensor& in, Tensor& out, double scale) {
  TORCH_CHECK(in.scalar_type() == at::kFloat && in.is_contiguous() && out.is_contiguous() && in.numel() == out.numel());
  chk_bf16(out, "out");
  c10::cuda::CUDAGuard guard(in.device());
  rb::cast_f32_to_bf16(in.data_ptr<float>(), out.data_ptr(), in.numel(), (float)scale, cur_stream());
}
void fill_uniform_hash(Tensor& out, int64_t seed, double bound) {
  chk_bf16(out, "out"); chk_2d_rowmajor(out, "out");
  c10::cuda::CUDAGuard guard(out.device());
  rb::fill_uniform_hash(out.data_ptr(), (int)out.size(0), (int)out.size(1), out.stride(0), (uint32_t)seed, (float)bound, cur_stream());
}
void seed_advance(Tensor& seed) {
  TORCH_CHECK(seed.is_cuda() && seed.scalar_type() == at::kInt && seed.numel() == 1);
  c10::cuda::CUDAGuard guard(seed.device());
  rb::seed_advance(reinterpret_cast<uint32_t*>(seed.data_ptr<int32_t>()), cur_stream());
}

void adamw_flat(Tensor& p, const Tensor& g, Tensor& m, Tensor& v, double lr, double b1, double b2, double eps, double wd, int64_t step,
                const OptTensor& grad_scale, double grad_scale_host, const OptTensor& skip, const OptTensor& step_dev) {
  chk_bf16(p, "param");
  TORCH_CHECK(p.is_contiguous() && g.is_contiguous() && m.is_contiguous() && v.is_contiguous());
  TORCH_CHECK(g.numel() == p.numel() && m.numel() == p.numel() && v.numel() == p.numel());
  const bool gf = g.scalar_type() == at::kFloat, sf = m.scalar_type() == at::kFloat;
  TORCH_CHECK(gf || g.scalar_type() == at::kBFloat16, "grad must be bf16 or fp32");
  TORCH_CHECK((sf || m.scalar_type() == at::kBFloat16) && m.scalar_type() == v.scalar_type(), "moments must be bf16 or fp32");
  c10::cuda::CUDAGuard guard(p.device());
  rb::adamw_flat(p.data_ptr(), g.data_ptr(), gf, m.data_ptr(), v.data_ptr(), sf, p.numel(), (float)lr, (float)b1, (float)b2, (float)eps,
                 (float)wd, (int)step, f32ptr(grad_scale), (float)grad_scale_host, f32ptr(skip), f32ptr(step_dev), cur_stream());
}
void sumsq(const Tensor& x, Tensor& out) {
  TORCH_CHECK(x.is_cuda() && x.is_contiguous() && out.scalar_type() == at::kFloat);
  const bool f = x.scalar_type() == at::kFloat;
  TORCH_CHECK(f || x.scalar_type() == at::kBFloat16);
  c10::cuda::CUDAGuard guard(x.device());
  rb::sumsq(x.data_ptr(), f, x.numel(), out.data_ptr<float>(), cur_stream());
}
void random_prune(Tensor& x, double ratio, int64_t seed, int64_t col_offset) {
  TORCH_CHECK(x.is_cuda() && x.is_contiguous());
  const bool f = x.scalar_type() == at::kFloat;
  TORCH_CHECK(f || x.scalar_type() == at::kBFloat16);
  c10::cuda::CUDAGuard guard(x.device());
  rb::random_prune(x.data_ptr(), f, x.numel(), (float)ratio, (uint32_t)seed, col_offset, cur_stream());
}
void magnitude_prune(Tensor& x, double ratio, Tensor& workspace, Tensor& thr) {
  TORCH_CHECK(x.is_cuda() && x.is_contiguous() && thr.scalar_type() == at::kFloat);
  TORCH_CHECK((size_t)workspace.numel() * workspace.element_size() >= rb::magnitude_quantile_workspace_bytes(), "workspace too small");
  const bool f = x.scalar_type() == at::kFloat;
  TORCH_CHECK(f || x.scalar_type() == at::kBFloat16);
  c10::cuda::CUDAGuard guard(x.device());
  rb::magnitude_quantile(x.data_ptr(), f, x.numel(), (float)ratio, thr.data_ptr<float>(), workspace.data_ptr(), cur_stream());
  rb::threshold_prune(x.data_ptr(), f, x.numel(), thr.data_ptr<float>(), cur_stream());
}

// ---------------------------------------------------------------------------------------------- NVLink collectives
rb::PeerPtrs peer_ptrs(const std::vector<int64_t>& v) {
  TORCH_CHECK((int)v.size() <= rb::kMaxPeers, "at most 8 peers");
  rb::PeerPtrs p;
  for (int i = 0; i < rb::kMaxPeers; ++i) p.ptr[i] = i < (int)v.size() ? reinterpret_cast<void*>(v[i]) : nullptr;
  return p;
}
rb::CommCtx comm_ctx(const std::vector<int64_t>& flag_ptrs, int64_t rank, int64_t world, Tensor& local_go) {
  TORCH_CHECK(local_go.is_cuda() && local_go.scalar_type() == at::kInt && local_go.numel() >= 2, "local_go must be int32[2] on the device");
  rb::CommCtx c;
  c.rank = (int)rank; c.world = (int)world; c.flags = peer_ptrs(flag_ptrs);
  c.local_go = reinterpret_cast<uint32_t*>(local_go.data_ptr<int32_t>());
  return c;
}
void comm_barrier(std::vector<int64_t> flag_ptrs, int64_t rank, int64_t world, Tensor& local_go, int64_t set, int64_t epoch) {
  c10::cuda::CUDAGuard guard(local_go.device());
  rb::xgpu_barrier(comm_ctx(flag_ptrs, rank, world, local_go), (int)set, (uint32_t)epoch, cur_stream());
}
void comm_allreduce_bf16(std::vector<int64_t> flag_ptrs, int64_t rank, int64_t world, Tensor& local_go, std::vector<int64_t> buf_ptrs,
                         int64_t mc_ptr, int64_t off_elems, int64_t n, int64_t epoch, int64_t max_blocks) {
  c10::cuda::CUDAGuard guard(local_go.device());
  rb::allreduce_bf16(comm_ctx(flag_ptrs, rank, world, local_go), peer_ptrs(buf_ptrs), reinterpret_cast<void*>(mc_ptr), off_elems, n,
                     (uint32_t)epoch, (int)max_blocks, cur_stream());
}
void comm_fused_update(std::vector<int64_t> flag_ptrs, int64_t rank, int64_t world, Tensor& local_go, const OptTensor& grads_f32,
                       std::vector<int64_t> grad_ptrs, int64_t grad_mc, Tensor& gred, std::vector<int64_t> param_ptrs, int64_t param_mc,
                       Tensor& exp_avg, Tensor& exp_avg_sq, int64_t n, double lr, double b1, double b2, double eps, double wd, int64_t step,
                       double max_norm, const OptTensor& skip, Tensor& norm_out, Tensor& scratch, int64_t epoch, int64_t max_blocks,
                       const OptTensor& step_dev, const OptTensor& loss_in, const OptTensor& loss_out) {
  if (grads_f32.has_value())
    TORCH_CHECK(grads_f32->scalar_type() == at::kFloat && grads_f32->is_contiguous() && grads_f32->numel() >= n, "grads must be fp32 [n]");
  TORCH_CHECK(gred.scalar_type() == at::kFloat && gred.numel() * world >= n, "gred must be fp32 [n / world]");
  chk_bf16(exp_avg, "exp_avg"); chk_bf16(exp_avg_sq, "exp_avg_sq");
  TORCH_CHECK(exp_avg.numel() * world >= n && exp_avg_sq.numel() * world >= n, "moments must be [n / world]");
  TORCH_CHECK(norm_out.scalar_type() == at::kFloat && scratch.scalar_type() == at::kFloat && scratch.numel() >= 3);
  c10::cuda::CUDAGuard guard(local_go.device());
  rb::FusedUpdateArgs a;
  a.grads_f32 = grads_f32.has_value() ? grads_f32->data_ptr<float>() : nullptr;
  a.grad_bufs = peer_ptrs(grad_ptrs); a.grad_mc = reinterpret_cast<void*>(grad_mc);
  a.gred = gred.data_ptr<float>();
  a.param_bufs = peer_ptrs(param_ptrs); a.param_mc = reinterpret_cast<void*>(param_mc);
  a.exp_avg = exp_avg.data_ptr(); a.exp_avg_sq = exp_avg_sq.data_ptr();
  a.n = n; a.lr = (float)lr; a.beta1 = (float)b1; a.beta2 = (float)b2; a.eps = (float)eps; a.weight_decay = (float)wd;
  a.step = (int)step; a.step_dev = f32ptr(step_dev); a.max_norm = (float)max_norm; a.inv_world = 1.0f / (float)world;
  a.loss_in = f32ptr(loss_in); a.loss_out = const_cast<float*>(f32ptr(loss_out));
  a.skip = f32ptr(skip); a.norm_out = norm_out.data_ptr<float>(); a.sq_accum = scratch.data_ptr<float>(); a.max_blocks = (int)max_blocks;
  rb::fused_update(comm_ctx(flag_ptrs, rank, world, local_go), a, (uint32_t)epoch, cur_stream());
}

long long launch_count() { return rb::g_launch_count; }
void reset_launch_count() { rb::g_launch_count = 0; }

}  // namespace

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "relora_b200 sm_100a kernels";
  m.def("gemm", &gemm, "tcgen05 GEMM with fused LoRA K-extension");
  m.def("gemm_clear_descriptor_cache", &rb::gemm_clear_descriptor_cache);
  m.def("gemm_pair_clusters", &rb::gemm_pair_clusters);
  m.def("gemm_set_trace", [](const OptTensor& t) {
    if (!t.has_value()) { rb::gemm_set_trace(nullptr); return; }
    TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kLong && t->is_contiguous() && t->numel() >= 16 * 512, "trace buffer: int64 CUDA tensor of >= 8192 elements");
    rb::gemm_set_trace(t->data_ptr());
  });
  m.def("rmsnorm_fwd", &rmsnorm_fwd, py::arg("x"), py::arg("w"), py::arg("y"), py::arg("rstd"), py::arg("eps"), py::arg("xd"), py::arg("seed"),
        py::arg("keys"), py::arg("p"), py::arg("q8") = py::none(), py::arg("q_inv_scale") = py::none(), py::arg("q_amax") = py::none());
  m.def("rmsnorm_bwd", &rmsnorm_bwd);
  m.def("rmsnorm_bwd_ws_blocks", &rb::rmsnorm_bwd_ws_blocks);
  m.def("dropout_expand", &dropout_expand, py::arg("x"), py::arg("xd"), py::arg("seed"), py::arg("keys"), py::arg("p"), py::arg("q8") = py::none(),
        py::arg("q_inv_scale") = py::none(), py::arg("q_amax") = py::none());
  m.def("dropout_combine", &dropout_combine);
  m.def("fp8_quantize_weight", &fp8_quantize_weight, py::arg("w"), py::arg("w8"), py::arg("scratch"), py::arg("scale"), py::arg("inv_scale"),
        py::arg("w8t") = py::none());
  m.def("fp8_quantize_act", &fp8_quantize_act, py::arg("x"), py::arg("x8"), py::arg("inv_scale"), py::arg("amax_cur") = py::none(), py::arg("e5m2") = false);
  m.def("fp8_prep", &fp8_prep, py::arg("state"), py::arg("w_scale"), py::arg("inv_sx"), py::arg("alpha_main"), py::arg("alpha_inv"), py::arg("margin"),
        py::arg("n_e4m3") = -1);
  m.def("attention_fwd", &attention_fwd);
  m.def("attention_occupancy", &rb::attention_occupancy);
  m.def("attention_set_trace", [](const OptTensor& t) {
    if (!t.has_value()) { rb::attention_set_trace(nullptr); return; }
    TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kLong && t->is_contiguous() && t->numel() >= 8 * 64, "trace buffer: int64 CUDA tensor of >= 512 elements");
    rb::attention_set_trace(t->data_ptr());
  });
  m.def("attention_bwd", &attention_bwd, py::arg("qkv"), py::arg("out"), py::arg("dout"), py::arg("lse"), py::arg("delta"), py::arg("dqkv"),
        py::arg("B"), py::arg("T"), py::arg("nh"), py::arg("hd"), py::arg("scale"), py::arg("ds_workspace") = py::none());
  m.def("attention_ds_workspace_elems", &rb::attention_ds_workspace_elems);
  m.def("lora_dx", &lora_dx, py::arg("dy"), py::arg("w"), py::arg("du"), py::arg("a"), py::arg("out"), py::arg("seed"), py::arg("keys"),
        py::arg("p"), py::arg("base") = py::none());
  m.def("rope_inplace", &rope_inplace);
  m.def("rope_pack_bwd", &rope_pack_bwd);
  m.def("swiglu_fwd", &swiglu_fwd, py::arg("gu"), py::arg("h"), py::arg("hd") = py::none(), py::arg("seed") = py::none(),
        py::arg("key") = 0, py::arg("p") = 0.0, py::arg("q8") = py::none(), py::arg("q_inv_scale") = py::none(), py::arg("q_amax") = py::none());
  m.def("swiglu_bwd", &swiglu_bwd);
  m.def("mx_sf_bytes", &mx_sf_bytes);
  m.def("mx_quantize_rows", &mx_quantize_rows);
  m.def("mx_quantize_weight_2d", &mx_quantize_weight_2d);
  m.def("mx_dequantize_weight", &mx_dequantize_weight);
  m.def("gemm_mx", &gemm_mx, py::arg("a"), py::arg("sfa"), py::arg("b"), py::arg("sfb"), py::arg("out"), py::arg("M"), py::arg("N"), py::arg("K"),
        py::arg("b_mn_major") = false, py::arg("a2") = py::none(), py::arg("b2") = py::none(), py::arg("residual") = py::none());
  m.def("layernorm_fwd", &layernorm_fwd);
  m.def("layernorm_bwd", &layernorm_bwd);
  m.def("gelu_fwd", &gelu_fwd);
  m.def("gelu_bwd", &gelu_bwd);
  m.def("neox_rope", &neox_rope);
  m.def("embedding_fwd", &embedding_fwd);
  m.def("embedding_bwd", &embedding_bwd);
  m.def("embedding_bwd_sorted", &embedding_bwd_sorted);
  m.def("cross_entropy_fwd_bwd", &cross_entropy_fwd_bwd);
  m.def("transpose", &transpose);
  m.def("add", &add);
  m.def("cast_f32_to_bf16", &cast_f32_to_bf16);
  m.def("fill_uniform_hash", &fill_uniform_hash);
  m.def("seed_advance", &seed_advance);
  m.def("adamw_flat", &adamw_flat);
  m.def("sumsq", &sumsq);
  m.def("random_prune", &random_prune);
  m.def("magnitude_prune", &magnitude_prune);
  m.def("quantile_workspace_bytes", &rb::magnitude_quantile_workspace_bytes);
  m.def("comm_barrier", &comm_barrier);
  m.def("comm_allreduce_bf16", &comm_allreduce_bf16);
  m.def("comm_fused_update", &comm_fused_update);
  m.def("launch_count", &launch_count);
  m.def("reset_launch_count", &reset_launch_count);
}
