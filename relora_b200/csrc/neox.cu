// Kernels of the GPT-NeoX / Pythia block that the Llama executor does not have (SURVEY K16):
//
//   layernorm_fwd / layernorm_bwd   nn.LayerNorm with affine weight + bias (reference modeling_pythia.py:413-414), warp per row,
//                                   fp32 statistics saved for the backward; dw / db accumulated through shared-memory block
//                                   partials and one 16-byte vector reduction per 4 columns per block
//   gelu_fwd / gelu_bwd             exact (erf) and tanh GELU (modeling_pythia.py:395-406), 128-bit accesses
//   neox_rope                       partial rotary embedding on the fused query_key_value output [rows, nh, 3*hd]
//                                   (q | k | v per head, first `rot` dims of q and k rotated, fp32 tables; :172-197), in place,
//                                   forward and inverse (backward) direction
#include "common.cuh"
#include "kernels.h"

namespace rb {

namespace {
constexpr int kRowsPerBlock = 8;  // one warp per row

template <int VPL>
__global__ void __launch_bounds__(kRowsPerBlock * 32) layernorm_fwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ w,
                                                                          const bf16* __restrict__ b, bf16* __restrict__ y,
                                                                          float* __restrict__ mean_out, float* __restrict__ rstd_out, int M,
                                                                          int H, float eps) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = blockIdx.x * kRowsPerBlock + warp;
  if (row >= M) return;
  const int nvec = H / 8;
  const uint4* xr = reinterpret_cast<const uint4*>(x + (long long)row * H);
  uint4 xv[VPL];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    if (c < nvec) {
      xv[i] = xr[c];
      float f[8];
      unpack8(xv[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += f[j];
    }
  }
  const float mean = warp_sum(s) / (float)H;
  float ss = 0.f;  // two-pass variance on the registers: no cancellation
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    if (c < nvec) {
      float f[8];
      unpack8(xv[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) ss += (f[j] - mean) * (f[j] - mean);
    }
  }
  const float rstd = rsqrtf(warp_sum(ss) / (float)H + eps);
  if (lane == 0) {
    mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
  uint4* yr = reinterpret_cast<uint4*>(y + (long long)row * H);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    if (c < nvec) {
      float f[8], wf[8], bf[8], o[8];
      unpack8(xv[i], f);
      unpack8(reinterpret_cast<const uint4*>(w)[c], wf);
      if (b != nullptr) unpack8(reinterpret_cast<const uint4*>(b)[c], bf);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (f[j] - mean) * rstd * wf[j] + (b != nullptr ? bf[j] : 0.f);
      yr[c] = pack8(o);
    }
  }
}

// dx = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * w;   dw += sum_rows dy * xhat;   db += sum_rows dy
template <int VPL>
__global__ void __launch_bounds__(kRowsPerBlock * 32) layernorm_bwd_kernel(const bf16* __restrict__ dy, const bf16* __restrict__ x,
                                                                          const bf16* __restrict__ w, const float* __restrict__ mean,
                                                                          const float* __restrict__ rstd, bf16* __restrict__ dx,
                                                                          float* __restrict__ dw, float* __restrict__ db, int M, int H) {
  extern __shared__ float sacc[];  // [2][H] block partials of dw, db
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nvec = H / 8;
  for (int c = threadIdx.x; c < 2 * H; c += blockDim.x) sacc[c] = 0.f;
  __syncthreads();
  uint4 wv[VPL];
  float dwacc[VPL][8], dbacc[VPL][8];
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    wv[i] = (c < nvec) ? reinterpret_cast<const uint4*>(w)[c] : make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int j = 0; j < 8; ++j) dwacc[i][j] = dbacc[i][j] = 0.f;
  }
  for (int row = blockIdx.x * kRowsPerBlock + warp; row < M; row += gridDim.x * kRowsPerBlock) {
    const float mu = mean[row], rs = rstd[row];
    uint4 dyv[VPL], xv[VPL];
    float sg = 0.f, sgx = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (c < nvec) {
        dyv[i] = reinterpret_cast<const uint4*>(dy + (long long)row * H)[c];
        xv[i] = reinterpret_cast<const uint4*>(x + (long long)row * H)[c];
        float dyf[8], xf[8], wf[8];
        unpack8(dyv[i], dyf);
        unpack8(xv[i], xf);
        unpack8(wv[i], wf);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float xh = (xf[j] - mu) * rs, g = dyf[j] * wf[j];
          sg += g;
          sgx += g * xh;
          dwacc[i][j] += dyf[j] * xh;
          dbacc[i][j] += dyf[j];
        }
      }
    }
    sg = warp_sum(sg) / (float)H;
    sgx = warp_sum(sgx) / (float)H;
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const int c = lane + i * 32;
      if (c < nvec) {
        float dyf[8], xf[8], wf[8], o[8];
        unpack8(dyv[i], dyf);
        unpack8(xv[i], xf);
        unpack8(wv[i], wf);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = rs * (dyf[j] * wf[j] - sg - (xf[j] - mu) * rs * sgx);
        reinterpret_cast<uint4*>(dx + (long long)row * H)[c] = pack8(o);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    const int c = lane + i * 32;
    if (c < nvec) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        atomicAdd(&sacc[c * 8 + j], dwacc[i][j]);
        atomicAdd(&sacc[H + c * 8 + j], dbacc[i][j]);
      }
    }
  }
  __syncthreads();
  for (int c = threadIdx.x * 4; c < H; c += blockDim.x * 4) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dw + c), "f"(sacc[c]), "f"(sacc[c + 1]), "f"(sacc[c + 2]), "f"(sacc[c + 3])
                 : "memory");
    if (db != nullptr)
      asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(db + c), "f"(sacc[H + c]), "f"(sacc[H + c + 1]), "f"(sacc[H + c + 2]),
                   "f"(sacc[H + c + 3])
                   : "memory");
  }
}

int pick_vpl(int nvec) {
  const int need = (nvec + 31) / 32;
  for (int v : {1, 2, 3, 4, 8, 16}) if (need <= v) return v;
  return 0;
}

__device__ __forceinline__ float gelu_erf(float z) { return 0.5f * z * (1.f + erff(z * 0.70710678118654752f)); }
__device__ __forceinline__ float dgelu_erf(float z) {
  return 0.5f * (1.f + erff(z * 0.70710678118654752f)) + z * 0.3989422804014327f * __expf(-0.5f * z * z);
}
__device__ __forceinline__ float gelu_tanh(float z) {
  const float u = 0.7978845608028654f * (z + 0.044715f * z * z * z);
  return 0.5f * z * (1.f + tanhf(u));
}
__device__ __forceinline__ float dgelu_tanh(float z) {
  const float u = 0.7978845608028654f * (z + 0.044715f * z * z * z), t = tanhf(u), sech2 = 1.f - t * t;
  // sech2 is exactly 0 once |u| > 9; skipping the term then keeps 0 * inf (z * z overflows above 1.8e19) from giving NaN
  return 0.5f * (1.f + t) + (sech2 > 0.f ? 0.5f * z * sech2 * 0.7978845608028654f * (1.f + 3.f * 0.044715f * z * z) : 0.f);
}

template <bool TANH>
__global__ void __launch_bounds__(256) gelu_fwd_kernel(const bf16* __restrict__ z, bf16* __restrict__ a, long long nvec) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float f[8];
    unpack8(reinterpret_cast<const uint4*>(z)[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = TANH ? gelu_tanh(f[j]) : gelu_erf(f[j]);
    reinterpret_cast<uint4*>(a)[i] = pack8(f);
  }
}
template <bool TANH>
__global__ void __launch_bounds__(256) gelu_bwd_kernel(const bf16* __restrict__ da, const bf16* __restrict__ z, bf16* __restrict__ dz,
                                                       long long nvec) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float g[8], f[8];
    unpack8(reinterpret_cast<const uint4*>(da)[i], g);
    unpack8(reinterpret_cast<const uint4*>(z)[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) g[j] *= TANH ? dgelu_tanh(f[j]) : dgelu_erf(f[j]);
    reinterpret_cast<uint4*>(dz)[i] = pack8(g);
  }
}

// one thread per (row, head, q|k, pair index i < rot/2): (a, b) = (x[i], x[i + rot/2]) -> (a cos - b sin, b cos + a sin)
__global__ void __launch_bounds__(256) neox_rope_kernel(bf16* __restrict__ qkv, long long ld, long long rows, int T, int nh, int hd, int rot,
                                                        const float* __restrict__ cos, const float* __restrict__ sin, int pos0, bool inverse) {
  const int half = rot / 2;
  const long long total = rows * nh * 2 * half;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = int(i % half);
    long long r = i / half;
    const int which = int(r % 2);  // 0 = q, 1 = k
    r /= 2;
    const int h = int(r % nh);
    const long long row = r / nh;
    const int pos = int(row % T) + pos0;
    bf16* base = qkv + row * ld + (long long)h * 3 * hd + which * hd;
    const float c = cos[(long long)pos * rot + p], s = inverse ? -sin[(long long)pos * rot + p] : sin[(long long)pos * rot + p];
    const float a = __bfloat162float(base[p]), b = __bfloat162float(base[p + half]);
    base[p] = __float2bfloat16_rn(a * c - b * s);
    base[p + half] = __float2bfloat16_rn(b * c + a * s);
  }
}
}  // namespace

bool layernorm_fwd(const void* x, const void* w, const void* b, void* y, float* mean, float* rstd, int M, int H, float eps, cudaStream_t s) {
  const int vpl = (H % 8 == 0) ? pick_vpl(H / 8) : 0;
  if (vpl == 0 || M <= 0) return false;
  const int grid = ceil_div(M, kRowsPerBlock);
  const bf16 *xp = (const bf16*)x, *wp = (const bf16*)w, *bp = (const bf16*)b;
#define L(V) launch_k(layernorm_fwd_kernel<V>, grid, kRowsPerBlock * 32, 0, s, xp, wp, bp, (bf16*)y, mean, rstd, M, H, eps)
  switch (vpl) {
    case 1: L(1); break;
    case 2: L(2); break;
    case 3: L(3); break;
    case 4: L(4); break;
    case 8: L(8); break;
    default: L(16); break;
  }
#undef L
  RB_CHECK_LAUNCH("layernorm_fwd");
  return true;
}

bool layernorm_bwd(const void* dy, const void* x, const void* w, const float* mean, const float* rstd, void* dx, float* dw, float* db, int M,
                   int H, cudaStream_t s) {
  const int vpl = (H % 8 == 0) ? pick_vpl(H / 8) : 0;
  if (vpl == 0 || vpl > 8 || M <= 0 || (reinterpret_cast<uintptr_t>(dw) & 15) != 0 || (db != nullptr && (reinterpret_cast<uintptr_t>(db) & 15) != 0))
    return false;
  const size_t smem = 2 * (size_t)H * sizeof(float);
  const int grid = std::min(ceil_div(M, kRowsPerBlock), 2 * num_sms());
  const bf16 *a = (const bf16*)dy, *bx = (const bf16*)x, *c = (const bf16*)w;
#define L(V) launch_k(layernorm_bwd_kernel<V>, grid, kRowsPerBlock * 32, smem, s, a, bx, c, mean, rstd, (bf16*)dx, dw, db, M, H)
  switch (vpl) {
    case 1: L(1); break;
    case 2: L(2); break;
    case 3: L(3); break;
    case 4: L(4); break;
    default: L(8); break;
  }
#undef L
  RB_CHECK_LAUNCH("layernorm_bwd");
  return true;
}

void gelu_fwd(const void* z, void* a, long long n, bool tanh_approx, cudaStream_t s) {
  if (n % 8) throw std::runtime_error("gelu: element count must be a multiple of 8");
  const long long nvec = n / 8;
  const int grid = (int)std::min<long long>((nvec + 255) / 256, (long long)num_sms() * 8);
  if (grid <= 0) return;
  if (tanh_approx) launch_k(gelu_fwd_kernel<true>, grid, 256, 0, s, (const bf16*)z, (bf16*)a, nvec);
  else launch_k(gelu_fwd_kernel<false>, grid, 256, 0, s, (const bf16*)z, (bf16*)a, nvec);
  RB_CHECK_LAUNCH("gelu_fwd");
}
void gelu_bwd(const void* da, const void* z, void* dz, long long n, bool tanh_approx, cudaStream_t s) {
  if (n % 8) throw std::runtime_error("gelu: element count must be a multiple of 8");
  const long long nvec = n / 8;
  const int grid = (int)std::min<long long>((nvec + 255) / 256, (long long)num_sms() * 8);
  if (grid <= 0) return;
  if (tanh_approx) launch_k(gelu_bwd_kernel<true>, grid, 256, 0, s, (const bf16*)da, (const bf16*)z, (bf16*)dz, nvec);
  else launch_k(gelu_bwd_kernel<false>, grid, 256, 0, s, (const bf16*)da, (const bf16*)z, (bf16*)dz, nvec);
  RB_CHECK_LAUNCH("gelu_bwd");
}

void neox_rope(void* qkv, long long ld, long long rows, int T, int nh, int hd, int rot, const float* cos, const float* sin, int pos0,
               bool inverse, cudaStream_t s) {
  if (rot <= 0) return;
  if (rot % 2 || rot > hd) throw std::runtime_error("neox_rope: rotary dims must be even and <= head_dim");
  const long long total = rows * nh * rot;  // 2 (q, k) * rot / 2 pairs
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)num_sms() * 16);
  if (grid <= 0) return;
  launch_k(neox_rope_kernel, grid, 256, 0, s, (bf16*)qkv, ld, rows, T, nh, hd, rot, cos, sin, pos0, inverse);
  RB_CHECK_LAUNCH("neox_rope");
}

}  // namespace rb
