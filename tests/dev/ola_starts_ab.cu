// A/B of the Hamming overlap-add at explicit starts (Roformer): the first form of ola_starts_kernel, a scan over all chunks per sample, against the
// binary-searched run of covering chunks it was replaced with.  Checks bit-identity and times both with CUDA events, alternating.
//   nvcc -O3 -gencode arch=compute_100a,code=sm_100a -o build/ola_starts_ab tests/dev/ola_starts_ab.cu && build/ola_starts_ab   (build/ is git-ignored)
#include <cstdio>
#include <cstdint>
#include <vector>
#include <cmath>
#include <algorithm>
#include <cuda_runtime.h>
__global__ void old_k(const float* __restrict__ chunks, const int64_t* __restrict__ starts, const float* __restrict__ window, int n_chunks, int channels, int len, int64_t n_out, float* __restrict__ out) {
  const int c = blockIdx.y;
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_out; q += (int64_t)gridDim.x * blockDim.x) {
    float acc = 0.f, cnt = 0.f;
    for (int i = 0; i < n_chunks; ++i) {
      const int64_t r = q - __ldg(&starts[i]);
      if (r >= 0 && r < len) { const float w = __ldg(&window[r]); acc = fmaf(__ldg(&chunks[((int64_t)i * channels + c) * len + r]), w, acc); cnt += w; }
    }
    out[(int64_t)c * n_out + q] = acc / fmaxf(cnt, 1e-10f);
  }
}
__device__ __forceinline__ int ub(const int64_t* __restrict__ a, int n, int64_t v) { int lo = 0, hi = n; while (lo < hi) { int m = (lo + hi) >> 1; if (__ldg(&a[m]) <= v) lo = m + 1; else hi = m; } return lo; }
__global__ void new_k(const float* __restrict__ chunks, const int64_t* __restrict__ starts, const float* __restrict__ window, int first, int n_local, int channels, int len, int64_t q_begin, int64_t q_end, float* __restrict__ out, int64_t out_ld, int64_t out_base) {
  const int c = blockIdx.y; const int64_t* st = starts + first;
  for (int64_t q = q_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < q_end; q += (int64_t)gridDim.x * blockDim.x) {
    float acc = 0.f, cnt = 0.f; const int i1 = ub(st, n_local, q);
    for (int i = ub(st, i1, q - len); i < i1; ++i) { const int64_t r = q - __ldg(&st[i]); const float w = __ldg(&window[r]); acc = fmaf(__ldg(&chunks[((int64_t)i * channels + c) * len + r]), w, acc); cnt += w; }
    out[(int64_t)c * out_ld + (q - out_base)] = acc / fmaxf(cnt, 1e-10f);
  }
}
__global__ void fill(float* x, int64_t n, uint32_t seed) { for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) { uint32_t h = (uint32_t)i * 2654435761u ^ seed; h ^= h >> 15; h *= 2246822519u; h ^= h >> 13; x[i] = (h & 0xffffff) / 16777216.f - 0.5f; } }
int main() {
  const int C = 441 * 800, SR = 44100, ch = 2;
  struct G { const char* name; int64_t N; int step; } grids[] = {{"ep_317 5-min overlap 8 (step = chunk)", 300LL * SR, C}, {"1-min overlap 0.03 (step 1323)", 60LL * SR, 1323}};
  for (auto g : grids) {
    std::vector<int64_t> st; for (int64_t i = 0; i < g.N; i += g.step) st.push_back(i + C <= g.N ? i : g.N - C);
    int n = (int)st.size();
    std::vector<float> hw(C); for (int m = 0; m < C; ++m) hw[m] = (float)(0.54 - 0.46 * cos(2.0 * M_PI * m / (C - 1)));
    float *ck, *w, *o1, *o2; int64_t* sd;
    cudaMalloc(&ck, (size_t)n * ch * C * 4); cudaMalloc(&w, C * 4); cudaMalloc(&o1, g.N * ch * 4); cudaMalloc(&o2, g.N * ch * 4); cudaMalloc(&sd, n * 8);
    cudaMemcpy(w, hw.data(), C * 4, cudaMemcpyHostToDevice); cudaMemcpy(sd, st.data(), n * 8, cudaMemcpyHostToDevice);
    fill<<<148 * 16, 256>>>(ck, (int64_t)n * ch * C, 7);
    dim3 grid((unsigned)std::min<int64_t>((g.N + 255) / 256, 148 * 8), ch);
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    float t_old = 0, t_new = 0; const int reps = 5;
    for (int r = 0; r < reps + 1; ++r) {  // alternate; first round is warm-up
      float a, b;
      cudaEventRecord(e0); old_k<<<grid, 256>>>(ck, sd, w, n, ch, C, g.N, o1); cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&a, e0, e1);
      cudaEventRecord(e0); new_k<<<grid, 256>>>(ck, sd, w, 0, n, ch, C, 0, g.N, o2, g.N, 0); cudaEventRecord(e1); cudaEventSynchronize(e1); cudaEventElapsedTime(&b, e0, e1);
      if (r) { t_old += a; t_new += b; }
    }
    std::vector<float> h1(g.N * ch), h2(g.N * ch);
    cudaMemcpy(h1.data(), o1, g.N * ch * 4, cudaMemcpyDeviceToHost); cudaMemcpy(h2.data(), o2, g.N * ch * 4, cudaMemcpyDeviceToHost);
    bool same = memcmp(h1.data(), h2.data(), h1.size() * 4) == 0;
    printf("{\"grid\": \"%s\", \"chunks\": %d, \"samples\": %lld, \"channels\": %d, \"old_scan_ms\": %.3f, \"new_search_ms\": %.3f, \"bit_identical\": %s, \"err\": \"%s\"}\n", g.name, n, (long long)g.N, ch,
           t_old / reps, t_new / reps, same ? "true" : "false", cudaGetErrorString(cudaGetLastError()));
    cudaFree(ck); cudaFree(w); cudaFree(o1); cudaFree(o2); cudaFree(sd);
  }
  return 0;
}
