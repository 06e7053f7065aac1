// Operators of the BS-Roformer path (uvr_lib_v5/roformer/bs_roformer.py, attend.py; the Roformer branch of mdxc_separator.py) that are
// not GEMMs: RMSNorm on (strided) rows, rotary embedding fused with the head split, sigmoid gating fused with the head merge, GLU over
// the last dimension into a column slice, the complex mask product that also re-orders to iSTFT planes, and the Hamming overlap-add
// with a weight counter at arbitrary chunk starts.
#include <math.h>

#include "common.cuh"

namespace b200sep {

// RMSNorm (bs_roformer.py:30-37): y = x / max(||x||_2, 1e-12) * sqrt(C) * gamma; one warp per row; rows may be column slices (ld_in / ld_out)
__global__ void rmsnorm_kernel(const float* __restrict__ x, const float* __restrict__ gamma, float* __restrict__ y, int64_t rows, int C, int64_t ld_in, int64_t ld_out) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float* xr = x + row * ld_in;
  float s = 0.f;
  for (int c = lane; c < C; c += 32) {
    const float v = xr[c];
    s = fmaf(v, v, s);
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float inv = sqrtf((float)C) / fmaxf(sqrtf(s), 1e-12f);
  float* yr = y + row * ld_out;
  for (int c = lane; c < C; c += 32) yr[c] = xr[c] * inv * __ldg(&gamma[c]);
}

// qkv (B, n, 3, H, dh) = the to_qkv output -> q, k, v (B, H, n, dh); q and k with the rotary embedding applied (positions 0..n-1, interleaved
// pairs, rotary-embedding-torch defaults).  One thread per (b, pos, h, pair): float2 loads and stores, all coalesced along d.
__global__ void rope_split_kernel(const float* __restrict__ qkv, const float* __restrict__ freqs, float* __restrict__ q, float* __restrict__ k, float* __restrict__ v,
                                  int n, int H, int dh, int64_t total) {
  const int half = dh >> 1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int p = (int)(i % half);
    const int h = (int)((i / half) % H);
    const int pos = (int)((i / ((int64_t)half * H)) % n);
    const int64_t b = i / ((int64_t)half * H * n);
    const float* src = qkv + ((b * n + pos) * 3) * (int64_t)H * dh + (int64_t)h * dh + 2 * p;
    float sn, cs;
    sincosf((float)pos * __ldg(&freqs[p]), &sn, &cs);
    const int64_t o = ((b * H + h) * n + pos) * (int64_t)dh + 2 * p;
    const float2 qv = *reinterpret_cast<const float2*>(src);
    const float2 kv = *reinterpret_cast<const float2*>(src + (int64_t)H * dh);
    const float2 vv = *reinterpret_cast<const float2*>(src + 2 * (int64_t)H * dh);
    *reinterpret_cast<float2*>(q + o) = make_float2(qv.x * cs - qv.y * sn, qv.y * cs + qv.x * sn);  // t*cos + rotate_half(t)*sin, rotate_half = (-x2, x1)
    *reinterpret_cast<float2*>(k + o) = make_float2(kv.x * cs - kv.y * sn, kv.y * cs + kv.x * sn);
    *reinterpret_cast<float2*>(v + o) = vv;
  }
}

// out (B, H, n, dh) * sigmoid(gates (B*n, H)) -> merged (B*n, H*dh)   (bs_roformer.py:78-81)
__global__ void gate_merge_kernel(const float* __restrict__ o, const float* __restrict__ gates, float* __restrict__ y, int n, int H, int dh, int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % dh);
    const int h = (int)((i / dh) % H);
    const int64_t bn = i / ((int64_t)dh * H);  // b*n + pos
    const int64_t b = bn / n, pos = bn - b * n;
    const float g = 1.f / (1.f + expf(-__ldg(&gates[bn * H + h])));
    y[i] = o[((b * H + h) * n + pos) * (int64_t)dh + d] * g;
  }
}

// nn.GLU(dim=-1) on rows (rows, 2C; ld_in) -> (rows, C) written at y with row stride ld_out (a column slice of the mask tensor)
__global__ void glu_rows_kernel(const float* __restrict__ a, float* __restrict__ y, int C, int64_t ld_in, int64_t ld_out, int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const int64_t r = i / C;
    const float u = a[r * ld_in + c], v = a[r * ld_in + C + c];
    y[r * ld_out + c] = u / (1.f + expf(-v));
  }
}

// stft (b, T, F, 4) [feature order (f, s, c)] x mask (b, n, T, F, 4) complex product per (f, s) -> iSTFT planes (b*n, 4, F, T)
// (bs_roformer.py:472-484: view_as_complex, multiply, "b n (f s) t -> (b n s) f t")
__global__ void mask_apply_kernel(const float* __restrict__ st, const float* __restrict__ mask, float* __restrict__ out, int n_stems, int T, int F, int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    // i indexes the OUTPUT (bn, s, f, t) so the stores coalesce along t
    const int t = (int)(i % T);
    const int f = (int)((i / T) % F);
    const int s = (int)((i / ((int64_t)T * F)) % 2);
    const int64_t bn = i / ((int64_t)T * F * 2);
    const int64_t b = bn / n_stems;
    const float* sp = st + ((b * T + t) * (int64_t)F + f) * 4 + 2 * s;
    const float* mp = mask + ((bn * T + t) * (int64_t)F + f) * 4 + 2 * s;
    const float xr = sp[0], xi = sp[1], mr = mp[0], mi = mp[1];
    const int64_t plane = (int64_t)F * T;
    float* op = out + (bn * 4 + 2 * s) * plane + (int64_t)f * T + t;
    op[0] = xr * mr - xi * mi;
    op[plane] = xr * mi + xi * mr;
  }
}

// Roformer branch of MDXCSeparator.demix (mdxc_separator.py:310-343): result += x * window; counter += window; result / clamp(counter, 1e-10)
// as a gather over the chunks covering each output sample.  chunks (n_local, channels, len) hold the global chunks [first, first + n_local); chunk i
// is placed at starts[i] (non-decreasing).  The chunks covering q are the contiguous index run with q - len < starts[i] <= q: two binary searches find
// it, and it is visited in ascending order, so every sample gets the contributions of a scan over all chunks in the same order.
__device__ __forceinline__ int upper_bound_i64(const int64_t* __restrict__ a, int n, int64_t v) {  // first index with a[i] > v
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(&a[mid]) <= v) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__global__ void ola_starts_kernel(const float* __restrict__ chunks, const int64_t* __restrict__ starts, const float* __restrict__ window, int first, int n_local,
                                  int channels, int len, int64_t q_begin, int64_t q_end, float* __restrict__ out, int64_t out_ld, int64_t out_base) {
  const int c = blockIdx.y;
  const int64_t* st = starts + first;
  for (int64_t q = q_begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < q_end; q += (int64_t)gridDim.x * blockDim.x) {
    float acc = 0.f, cnt = 0.f;
    const int i1 = upper_bound_i64(st, n_local, q);
    for (int i = upper_bound_i64(st, i1, q - len); i < i1; ++i) {
      const int64_t r = q - __ldg(&st[i]);
      const float w = __ldg(&window[r]);
      acc = fmaf(__ldg(&chunks[((int64_t)i * channels + c) * len + r]), w, acc);
      cnt += w;
    }
    out[(int64_t)c * out_ld + (q - out_base)] = acc / fmaxf(cnt, 1e-10f);
  }
}

// Mel-Band Roformer (mel_band_roformer.py:300-303): x[row][g] = src[row][idx[g]] for (re, im) pairs; row = (b, t)
__global__ void gather_pairs_kernel(const float2* __restrict__ src, const int* __restrict__ idx, float2* __restrict__ dst, int n_src, int G, int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int g = (int)(i % G);
    const int64_t row = i / G;
    dst[i] = src[row * n_src + __ldg(&idx[g])];
  }
}

// masks_summed / num_bands_per_freq (mel_band_roformer.py:306-318) as a gather on the output side: for every (row, fs) the complex masks of the
// bands covering that frequency (CSR list of positions in the gathered axis) are summed and divided by their count.
__global__ void mask_average_kernel(const float2* __restrict__ mg, const int* __restrict__ off, const int* __restrict__ pos, float2* __restrict__ out, int G, int FS,
                                    int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int fs = (int)(i % FS);
    const int64_t row = i / FS;
    const int a = __ldg(&off[fs]), b = __ldg(&off[fs + 1]);
    float2 acc = make_float2(0.f, 0.f);
    for (int e = a; e < b; ++e) {
      const float2 v = mg[row * G + __ldg(&pos[e])];
      acc.x += v.x;
      acc.y += v.y;
    }
    const float inv = 1.f / fmaxf((float)(b - a), 1e-8f);
    out[i] = make_float2(acc.x * inv, acc.y * inv);
  }
}

static inline int rf_grid(int64_t n) { return (int)std::min<int64_t>(cdiv(n, 256), kNumSMs * 16); }

}  // namespace b200sep

using namespace b200sep;

extern "C" int b200sep_rmsnorm_f32(const float* x, const float* gamma, float* y, int64_t rows, int C, int64_t ld_in, int64_t ld_out, void* stream) {
  B2_CHECK_ARG(x && gamma && y && rows >= 0 && C >= 1 && ld_in >= C && ld_out >= C, "rmsnorm_f32: bad argument");
  if (rows == 0) return B200SEP_OK;
  rmsnorm_kernel<<<(unsigned)cdiv(rows, 8), 256, 0, (cudaStream_t)stream>>>(x, gamma, y, rows, C, ld_in, ld_out);
  B2_LAUNCHED();
  return B200SEP_OK;
}

extern "C" int b200sep_rope_split_heads_f32(const float* qkv, const float* freqs, float* q, float* k, float* v, int B, int n, int H, int dh, void* stream) {
  B2_CHECK_ARG(qkv && freqs && q && k && v && B >= 1 && n >= 1 && H >= 1 && dh >= 2 && dh % 2 == 0, "rope_split_heads_f32: bad argument");
  B2_CHECK_ARG(((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v)) & 7) == 0,
               "rope_split_heads_f32: buffers must be 8-byte aligned");
  const int64_t total = (int64_t)B * n * H * (dh / 2);
  rope_split_kernel<<<rf_grid(total), 256, 0, (cudaStream_t)stream>>>(qkv, freqs, q, k, v, n, H, dh, total);
  B2_LAUNCHED();
  return B200SEP_OK;
}

// float4 variant (dh % 4 == 0): one thread per four consecutive d
__global__ void gate_merge_vec_kernel(const float4* __restrict__ o, const float* __restrict__ gates, float4* __restrict__ y, int n, int H, int dhq, int64_t total) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int d = (int)(i % dhq);
    const int h = (int)((i / dhq) % H);
    const int64_t bn = i / ((int64_t)dhq * H);
    const int64_t b = bn / n, pos = bn - b * n;
    const float g = 1.f / (1.f + expf(-__ldg(&gates[bn * H + h])));
    const float4 v = o[((b * H + h) * n + pos) * (int64_t)dhq + d];
    y[i] = make_float4(v.x * g, v.y * g, v.z * g, v.w * g);
  }
}

extern "C" int b200sep_gate_merge_heads_f32(const float* o, const float* gates, float* y, int B, int n, int H, int dh, void* stream) {
  B2_CHECK_ARG(o && gates && y && B >= 1 && n >= 1 && H >= 1 && dh >= 1, "gate_merge_heads_f32: bad argument");
  if (dh % 4 == 0 && ((reinterpret_cast<uintptr_t>(o) | reinterpret_cast<uintptr_t>(y)) & 15) == 0) {
    const int64_t tq = (int64_t)B * n * H * (dh / 4);
    gate_merge_vec_kernel<<<rf_grid(tq), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float4*>(o), gates, reinterpret_cast<float4*>(y), n, H, dh / 4, tq);
    B2_LAUNCHED();
    return B200SEP_OK;
  }
  const int64_t total = (int64_t)B * n * H * dh;
  gate_merge_kernel<<<rf_grid(total), 256, 0, (cudaStream_t)stream>>>(o, gates, y, n, H, dh, total);
  B2_LAUNCHED();
  return B200SEP_OK;
}

extern "C" int b200sep_glu_rows_f32(const float* a, float* y, int64_t rows, int C, int64_t ld_in, int64_t ld_out, void* stream) {
  B2_CHECK_ARG(a && y && rows >= 0 && C >= 1 && ld_in >= 2 * C && ld_out >= C, "glu_rows_f32: bad argument");
  const int64_t total = rows * C;
  if (total == 0) return B200SEP_OK;
  glu_rows_kernel<<<rf_grid(total), 256, 0, (cudaStream_t)stream>>>(a, y, C, ld_in, ld_out, total);
  B2_LAUNCHED();
  return B200SEP_OK;
}

extern "C" int b200sep_roformer_mask_apply(const float* stft_tf, const float* mask, float* planes, int B, int n_stems, int T, int F, void* stream) {
  B2_CHECK_ARG(stft_tf && mask && planes && B >= 1 && n_stems >= 1 && T >= 1 && F >= 1, "roformer_mask_apply: bad argument");
  const int64_t total = (int64_t)B * n_stems * 2 * F * T;
  mask_apply_kernel<<<rf_grid(total), 256, 0, (cudaStream_t)stream>>>(stft_tf, mask, planes, n_stems, T, F, total);
  B2_LAUNCHED();
  return B200SEP_OK;
}

extern "C" int b200sep_overlap_add_starts_range(const float* chunks, const int64_t* starts, const float* window, int first, int n_local, int n_chunks, int channels,
                                                int len, int64_t n_out, int64_t q_begin, int64_t q_end, float* out, int64_t out_ld, int64_t out_base, void* stream) {
  B2_CHECK_ARG(chunks && starts && window && out && n_chunks >= 1 && channels >= 1 && len >= 1 && n_out >= 1, "overlap_add_starts: bad argument");
  B2_CHECK_ARG(0 <= first && n_local >= 1 && (int64_t)first + n_local <= n_chunks, "overlap_add_starts: local chunks [%d, %d) are not a run of the %d chunks", first,
               first + n_local, n_chunks);
  B2_CHECK_ARG(0 <= q_begin && q_begin <= q_end && q_end <= n_out, "overlap_add_starts: bad output range");
  B2_CHECK_ARG(out_base >= 0 && out_base <= q_begin && q_end - out_base <= out_ld, "overlap_add_starts: output slice does not cover [%lld, %lld)", (long long)q_begin,
               (long long)q_end);
  if (q_end == q_begin) return B200SEP_OK;
  if (first > 0 || first + n_local < n_chunks) {
    // every chunk covering [q_begin, q_end) must be local: the chunk before the run ends at or before q_begin, the one after it starts at or after
    // q_end.  The start list lives on the device; its two boundary entries are read back (a stream synchronisation, sharded calls only).
    int64_t edge[2] = {INT64_MIN, INT64_MAX};
    cudaStream_t s = (cudaStream_t)stream;
    if (first > 0) B2_CUDA(cudaMemcpyAsync(&edge[0], starts + first - 1, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    if (first + n_local < n_chunks) B2_CUDA(cudaMemcpyAsync(&edge[1], starts + first + n_local, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    B2_CUDA(cudaStreamSynchronize(s));
    B2_CHECK_ARG((first == 0 || edge[0] + len <= q_begin) && (first + n_local == n_chunks || edge[1] >= q_end),
                 "overlap_add_starts: outputs [%lld,%lld) need chunks outside the buffer's [%d,%d) (chunk %d starts at %lld, chunk %d at %lld)", (long long)q_begin,
                 (long long)q_end, first, first + n_local, first - 1, (long long)edge[0], first + n_local, (long long)edge[1]);
  }
  dim3 grid((unsigned)std::min<int64_t>(cdiv(q_end - q_begin, 256), kNumSMs * 8), channels);
  ola_starts_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(chunks, starts, window, first, n_local, channels, len, q_begin, q_end, out, out_ld, out_base);
  B2_LAUNCHED();
  return B200SEP_OK;
}

extern "C" int b200sep_overlap_add_starts(const float* chunks, const int64_t* starts, const float* window, int n_chunks, int channels, int len, int64_t n_out, float* out,
                                          void* stream) {
  return b200sep_overlap_add_starts_range(chunks, starts, window, 0, n_chunks, n_chunks, channels, len, n_out, 0, n_out, out, n_out, 0, stream);
}

extern "C" int b200sep_gather_pairs_f32(const float* src, const int* idx, float* dst, int64_t rows, int n_src_pairs, int n_gather, void* stream) {
  B2_CHECK_ARG(src && idx && dst && rows >= 0 && n_src_pairs >= 1 && n_gather >= 1, "gather_pairs_f32: bad argument");
  const int64_t total = rows * n_gather;
  if (total == 0) return B200SEP_OK;
  gather_pairs_kernel<<<rf_grid(total), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float2*>(src), idx, reinterpret_cast<float2*>(dst), n_src_pairs, n_gather, total);
  B2_LAUNCHED();
  return B200SEP_OK;
}

extern "C" int b200sep_mask_average_f32(const float* mask_gathered, const int* csr_offsets, const int* csr_positions, float* mask_out, int64_t rows, int n_gather, int n_out,
                                        void* stream) {
  B2_CHECK_ARG(mask_gathered && csr_offsets && csr_positions && mask_out && rows >= 0 && n_gather >= 1 && n_out >= 1, "mask_average_f32: bad argument");
  const int64_t total = rows * n_out;
  if (total == 0) return B200SEP_OK;
  mask_average_kernel<<<rf_grid(total), 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const float2*>(mask_gathered), csr_offsets, csr_positions,
                                                                        reinterpret_cast<float2*>(mask_out), n_gather, n_out, total);
  B2_LAUNCHED();
  return B200SEP_OK;
}
