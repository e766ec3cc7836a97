// E4M3 quantisation for the fp8 frozen-weight path (tcgen05 kind::f8f6f4 GEMMs, csrc/gemm_tcgen05.cu).
// Capability being replaced: the reference's bitsandbytes-quantised frozen weights (peft_pretraining/relora.py:224-236,
// 277-299, 314-317: NF4 / int8 storage, dequantise -> bf16 matmul); here the frozen GEMMs themselves run in fp8.
//
//   weights     : per-tensor scale from the current amax, refreshed at every ReLoRA merge
//   activations : per-tensor *delayed* scaling: a site quantises with the scale derived from the amax it observed in the
//                 previous micro-step and records the current amax for the next one (fp8_prep rotates the state)
// x ≈ s_x · q_x, W ≈ s_w · q_W  =>  x·Wᵀ = (s_x s_w) · Σ q_x q_W; the product scale reaches the GEMM epilogue as a device scalar.
#include <cuda_fp8.h>

#include "common.cuh"
#include "kernels.h"

namespace rb {

namespace {

constexpr float kE4M3Max = 448.f;

__device__ __forceinline__ void atomic_max_nonneg(float* addr, float v) {  // v >= 0: integer order == float order
  atomicMax(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__global__ void __launch_bounds__(256) amax_kernel(const bf16* __restrict__ x, long long ld, int R, int C, float* __restrict__ amax) {
  const int cv = C / 8;
  const long long total = (long long)R * cv;
  float m = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cv;
    const int c = int(i % cv) * 8;
    float f[8];
    unpack8(*reinterpret_cast<const uint4*>(x + r * ld + c), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(f[j]));
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) atomic_max_nonneg(amax, m);
}

// out = sat_fp8(x * inv_scale) (E4M3, or E5M2 for gradients); optionally records amax(|x|) into *amax_cur
template <bool E5M2>
__global__ void __launch_bounds__(256) quantize_kernel(const bf16* __restrict__ x, long long ld, uint8_t* __restrict__ out, long long ld8,
                                                       int R, int C, const float* __restrict__ inv_scale, float* __restrict__ amax_cur) {
  pdl_wait();
  pdl_launch_dependents();
  const float inv = *inv_scale;
  const int cv = C / 16;
  const long long total = (long long)R * cv;
  float m = 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / cv;
    const int c = int(i % cv) * 16;
    float f[16], lo8[8], hi8[8];
    unpack8(*reinterpret_cast<const uint4*>(x + r * ld + c), lo8);
    unpack8(*reinterpret_cast<const uint4*>(x + r * ld + c + 8), hi8);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      f[j] = lo8[j];
      f[8 + j] = hi8[j];
    }
    uint32_t w[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
      for (int j = 0; j < 4; ++j) m = fmaxf(m, fabsf(f[q * 4 + j]));
      const __nv_fp8x2_storage_t lo = __nv_cvt_float2_to_fp8x2(make_float2(f[q * 4] * inv, f[q * 4 + 1] * inv), __NV_SATFINITE, E5M2 ? __NV_E5M2 : __NV_E4M3);
      const __nv_fp8x2_storage_t hi = __nv_cvt_float2_to_fp8x2(make_float2(f[q * 4 + 2] * inv, f[q * 4 + 3] * inv), __NV_SATFINITE, E5M2 ? __NV_E5M2 : __NV_E4M3);
      w[q] = (uint32_t)lo | ((uint32_t)hi << 16);
    }
    *reinterpret_cast<uint4*>(out + r * ld8 + c) = make_uint4(w[0], w[1], w[2], w[3]);
  }
  if (amax_cur != nullptr) {
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) atomic_max_nonneg(amax_cur, m);
  }
}

// w8t[c, r] = sat_e4m3(w[r, c] * inv_scale): E4M3 copy of Wᵀ, the K-major operand of the input-gradient GEMM dy·W
__global__ void __launch_bounds__(256) quantize_transpose_kernel(const bf16* __restrict__ w, long long ld, uint8_t* __restrict__ out,
                                                                 long long ld8, int R, int C, const float* __restrict__ inv_scale) {
  __shared__ float tile[32][33];
  const float inv = *inv_scale;
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int j = ty; j < 32; j += 8) {
    const int r = r0 + j, c = c0 + tx;
    tile[j][tx] = (r < R && c < C) ? __bfloat162float(w[(long long)r * ld + c]) : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j, r = r0 + tx;
    if (c < C && r < R)
      out[(long long)c * ld8 + r] = (uint8_t)__nv_cvt_float_to_fp8(tile[tx][j] * inv, __NV_SATFINITE, __NV_E4M3);
  }
}

__global__ void weight_scale_kernel(const float* __restrict__ amax, float* __restrict__ scale, float* __restrict__ inv_scale) {
  const float s = fmaxf(*amax, 1e-12f) / kE4M3Max;
  *scale = s;
  *inv_scale = 1.0f / s;
}

// per activation site i: state[i] = {amax of the previous micro-step, amax being recorded}
__global__ void prep_kernel(float* __restrict__ state, const float* __restrict__ w_scale, float* __restrict__ inv_sx,
                            float* __restrict__ alpha_main, float* __restrict__ alpha_inv, int n, float margin, int n_e4m3) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float fmax = i < n_e4m3 ? kE4M3Max : 57344.f;  // sites >= n_e4m3 are gradients quantised to E5M2
  const float cur = state[2 * i + 1];
  // nothing recorded yet, or an overflowed activation (inf; NaN fails the comparison too): keep the old estimate
  const float prev = (isfinite(cur) && cur > 0.f) ? cur : state[2 * i];
  state[2 * i] = prev;
  state[2 * i + 1] = 0.f;
  const float sx = fmaxf(prev, 1e-12f) * margin / fmax;
  inv_sx[i] = 1.0f / sx;
  const float a = sx * w_scale[i];
  alpha_main[i] = a;
  alpha_inv[i] = 1.0f / a;
}

int grid_for(long long total) { return (int)std::max<long long>(1, std::min<long long>((total + 255) / 256, (long long)num_sms() * 8)); }

}  // namespace

void fp8_quantize_weight(const void* w, long long ld, void* w8, long long ld8, void* w8t, long long ld8t, int R, int C,
                         float* amax_scratch, float* scale, float* inv_scale, cudaStream_t s) {
  if (C % 16 != 0 || ld % 8 != 0 || ld8 % 16 != 0) throw std::runtime_error("fp8_quantize_weight: columns must be a multiple of 16");
  check(cudaMemsetAsync(amax_scratch, 0, sizeof(float), s), "cudaMemsetAsync(amax)");
  amax_kernel<<<grid_for((long long)R * C / 8), 256, 0, s>>>((const bf16*)w, ld, R, C, amax_scratch);
  RB_CHECK_LAUNCH("fp8_amax");
  weight_scale_kernel<<<1, 1, 0, s>>>(amax_scratch, scale, inv_scale);
  RB_CHECK_LAUNCH("fp8_weight_scale");
  quantize_kernel<false><<<grid_for((long long)R * C / 16), 256, 0, s>>>((const bf16*)w, ld, (uint8_t*)w8, ld8, R, C, inv_scale, nullptr);
  RB_CHECK_LAUNCH("fp8_quantize");
  if (w8t != nullptr) {
    dim3 grid((C + 31) / 32, (R + 31) / 32);
    quantize_transpose_kernel<<<grid, 256, 0, s>>>((const bf16*)w, ld, (uint8_t*)w8t, ld8t, R, C, inv_scale);
    RB_CHECK_LAUNCH("fp8_quantize_transpose");
  }
}

void fp8_quantize_act(const void* x, long long ld, void* x8, long long ld8, int R, int C, const float* inv_scale, float* amax_cur,
                      bool e5m2, cudaStream_t s) {
  if (C % 16 != 0 || ld % 8 != 0 || ld8 % 16 != 0) throw std::runtime_error("fp8_quantize_act: columns must be a multiple of 16");
  if (e5m2) launch_k(quantize_kernel<true>, grid_for((long long)R * C / 16), 256, 0, s, (const bf16*)x, ld, (uint8_t*)x8, ld8, R, C, inv_scale, amax_cur);
  else launch_k(quantize_kernel<false>, grid_for((long long)R * C / 16), 256, 0, s, (const bf16*)x, ld, (uint8_t*)x8, ld8, R, C, inv_scale, amax_cur);
  RB_CHECK_LAUNCH("fp8_quantize_act");
}

void fp8_prep(float* state, const float* w_scale, float* inv_sx, float* alpha_main, float* alpha_inv, int n, float margin,
              int n_e4m3, cudaStream_t s) {
  launch_k(prep_kernel, (n + 127) / 128, 128, 0, s, state, w_scale, inv_sx, alpha_main, alpha_inv, n, margin, n_e4m3);
  RB_CHECK_LAUNCH("fp8_prep");
}

}  // namespace rb
