// Element-wise / reduction kernels on pair tensors (see elementwise.cuh).  All HBM-bound: one pass over the plane for the
// mean, one for the centred second moment and one to apply (passes 2 and 3 re-read the 0.5-1 MB plane from L2).
#include "elementwise.cuh"

#include <cuda_bf16.h>

#include "umma_ops.cuh"  // split_pair / join_pair (self-test)

namespace b200sep {

using bf16 = __nv_bfloat16;

__device__ __forceinline__ float block_sum(float v, float* red) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  float t = (threadIdx.x < nw) ? red[threadIdx.x] : 0.f;
  if (w == 0) {
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (l == 0) red[0] = t;
  }
  __syncthreads();
  return red[0];
}

__device__ __forceinline__ void load8(const bf16* hi, const bf16* lo, int64_t i, float* v) {
  const uint4 h = __ldg(reinterpret_cast<const uint4*>(hi + i)), l = __ldg(reinterpret_cast<const uint4*>(lo + i));
  const bf16* hp = reinterpret_cast<const bf16*>(&h);
  const bf16* lp = reinterpret_cast<const bf16*>(&l);
#pragma unroll
  for (int k = 0; k < 8; ++k) v[k] = __bfloat162float(hp[k]) + __bfloat162float(lp[k]);
}

// grid (C, B), one CTA per plane; P % 8 == 0
__global__ void __launch_bounds__(512) instnorm_act_kernel(const bf16* __restrict__ x_hi, const bf16* __restrict__ x_lo, int x_c_total, int x_c_off,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta, int act, bf16* __restrict__ y_hi,
                                                          bf16* __restrict__ y_lo, int C, int64_t P) {
  __shared__ float red[32];
  const int c = blockIdx.x, b = blockIdx.y;
  const int64_t xo = ((int64_t)b * x_c_total + x_c_off + c) * P, yo = ((int64_t)b * C + c) * P;
  float s = 0.f;
  for (int64_t i = (int64_t)threadIdx.x * 8; i < P; i += (int64_t)blockDim.x * 8) {
    float v[8];
    load8(x_hi + xo, x_lo + xo, i, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) s += v[k];
  }
  const float mean = block_sum(s, red) / (float)P;
  float q = 0.f;
  for (int64_t i = (int64_t)threadIdx.x * 8; i < P; i += (int64_t)blockDim.x * 8) {
    float v[8];
    load8(x_hi + xo, x_lo + xo, i, v);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const float d = v[k] - mean;
      q = fmaf(d, d, q);
    }
  }
  const float var = block_sum(q, red) / (float)P;  // biased, like F.instance_norm
  const float rstd = rsqrtf(var + 1e-5f);
  const float g = __ldg(&gamma[c]) * rstd, bb = __ldg(&beta[c]);
  for (int64_t i = (int64_t)threadIdx.x * 8; i < P; i += (int64_t)blockDim.x * 8) {
    float v[8];
    load8(x_hi + xo, x_lo + xo, i, v);
    __align__(16) bf16 h[8];
    __align__(16) bf16 l[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float y = fmaf(v[k] - mean, g, bb);
      if (act == 2) y = 0.5f * y * (1.f + erff(y * 0.70710678118654752440f));
      else if (act == 1) y = fmaxf(y, 0.f);
      h[k] = __float2bfloat16_rn(y);
      l[k] = __float2bfloat16_rn(y - __bfloat162float(h[k]));
    }
    *reinterpret_cast<uint4*>(y_hi + yo + i) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint4*>(y_lo + yo + i) = *reinterpret_cast<const uint4*>(l);
  }
}

int instnorm_act_pair(const void* x_hi, const void* x_lo, int x_c_total, int x_c_off, const float* gamma, const float* beta, int act, void* y_hi, void* y_lo, int B,
                      int C, int64_t P, cudaStream_t st) {
  B2_CHECK_ARG(P % 8 == 0 && B >= 1 && C >= 1 && B <= 65535, "instnorm_act_pair: plane size %lld must be a multiple of 8", (long long)P);
  dim3 grid(C, B);
  instnorm_act_kernel<<<grid, 512, 0, st>>>((const bf16*)x_hi, (const bf16*)x_lo, x_c_total, x_c_off, gamma, beta, act, (bf16*)y_hi, (bf16*)y_lo, C, P);
  B2_LAUNCHED();
  return B200SEP_OK;
}

__global__ void cws_split_kernel(const float* __restrict__ spec, bf16* __restrict__ y_hi, bf16* __restrict__ y_lo, int Cc, int T, int K, int Fs, int c_total, int c_off,
                                 int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    // i enumerates the OUTPUT (b, c*K+k, t, f')
    const int f = (int)(i % Fs);
    int64_t r = i / Fs;
    const int t = (int)(r % T);
    r /= T;
    const int ck = (int)(r % (Cc * K));
    const int b = (int)(r / (Cc * K));
    const int c = ck / K, k = ck - c * K;
    const float v = __ldg(&spec[(((int64_t)b * Cc + c) * T + t) * ((int64_t)K * Fs) + (int64_t)k * Fs + f]);
    const int64_t o = (((int64_t)b * c_total + c_off + ck) * T + t) * Fs + f;
    const bf16 h = __float2bfloat16_rn(v);
    y_hi[o] = h;
    y_lo[o] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}
int cws_split_pair(const float* spec, void* y_hi, void* y_lo, int B, int Cc, int T, int K, int Fs, int c_total, int c_off, cudaStream_t st) {
  const int64_t n = (int64_t)B * Cc * K * T * Fs;
  if (n == 0) return B200SEP_OK;
  cws_split_kernel<<<(int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 16), 256, 0, st>>>(spec, (bf16*)y_hi, (bf16*)y_lo, Cc, T, K, Fs, c_total, c_off, n);
  B2_LAUNCHED();
  return B200SEP_OK;
}

__global__ void cws_merge_kernel(const float* __restrict__ x, float* __restrict__ spec, int S, int Cc, int T, int K, int Fs, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    // i enumerates the INPUT (b, (s*Cc + c)*K + k, t, f')
    const int f = (int)(i % Fs);
    int64_t r = i / Fs;
    const int t = (int)(r % T);
    r /= T;
    const int k = (int)(r % K);
    r /= K;
    const int c = (int)(r % Cc);
    r /= Cc;
    const int s = (int)(r % S);
    const int b = (int)(r / S);
    spec[((((int64_t)b * S + s) * Cc + c) * T + t) * ((int64_t)K * Fs) + (int64_t)k * Fs + f] = x[i];
  }
}
int cws_merge_f32(const float* x, float* spec, int B, int S, int Cc, int T, int K, int Fs, cudaStream_t st) {
  const int64_t n = (int64_t)B * S * Cc * K * T * Fs;
  if (n == 0) return B200SEP_OK;
  cws_merge_kernel<<<(int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 16), 256, 0, st>>>(x, spec, S, Cc, T, K, Fs, n);
  B2_LAUNCHED();
  return B200SEP_OK;
}

}  // namespace b200sep

// ---------------------------------------------------------------------------------------------------------
// self-test entry point (C ABI): fp32 in -> split -> instnorm_act_pair -> join -> fp32 out, synchronous
using namespace b200sep;

extern "C" int b200sep_selftest_instnorm_act(const float* x, const float* gamma, const float* beta, float* out, int B, int C, int x_c_total, int x_c_off, int64_t P,
                                             int act, void* stream) {
  B2_CHECK_ARG(x && gamma && beta && out, "selftest_instnorm_act: NULL argument");
  B2_CHECK_ARG(x_c_off >= 0 && x_c_off + C <= x_c_total && act >= 0 && act <= 2, "selftest_instnorm_act: channels [%d, %d) of %d / act=%d", x_c_off, x_c_off + C,
               x_c_total, act);
  cudaStream_t st = (cudaStream_t)stream;
  uint16_t *x_p = nullptr, *y_p = nullptr;
  const int64_t nx = (int64_t)B * x_c_total * P, ny = (int64_t)B * C * P;
  B2_CUDA(cudaMalloc(&x_p, nx * 4));
  B2_CUDA(cudaMalloc(&y_p, ny * 4));
  int rc = split_pair(x, x_p, x_p + nx, nx, st);
  if (!rc) rc = instnorm_act_pair(x_p, x_p + nx, x_c_total, x_c_off, gamma, beta, act, y_p, y_p + ny, B, C, P, st);
  if (!rc) rc = join_pair(y_p, y_p + ny, out, ny, st);
  cudaStreamSynchronize(st);
  cudaFree(x_p); cudaFree(y_p);
  return rc;
}
