// tcgen05 tensor-core operators on "pair" tensors (fp32 values stored as two bf16 planes, hi + lo).
//
// Why pairs: the reference computes the networks in fp32 and parity is gated at 1e-4 on PCM samples; a single
// TF32/BF16 pass misses that (measured 5e-4 / 3e-3 relative on the ConvTDFNet), so every contraction is evaluated as
//      A*B ~= Ah*Bh + Ah*Bl + Al*Bh          (Ah = bf16(A), Al = bf16(A - Ah); dropped terms <= 2^-16 |A||B|)
// with fp32 accumulation in TMEM: three kind::f16 UMMAs per k-step at the bf16 rate (measured error 7e-6 relative,
// DESIGN.md).  Producers write activations already split, so a pair tensor costs the same 4 bytes/element as fp32
// and its planes are fed to the tensor cores straight from TMA-written shared memory, no register staging.
//
// One kernel, two addressing modes:
//   GEMM : D[M][N] = A[M][K] * W[N][K]^T     (TDF linears; A, W K-major, TMA SWIZZLE_128B tiles of 64 k)
//   CONV : implicit GEMM for the 3x3 stride-1 convolution on (B,C,T,F) pairs.  The A tile of one filter ROW dy is a
//          TMA box [kc channels][128 pixels along F] at row t+dy-1 (out-of-bounds rows zero-filled = the padding); it
//          lands MN-major (pixels contiguous), which tcgen05 consumes directly (a_major = MN).  TMA cannot shift a box
//          by one bf16 along the innermost axis (box starts must be 16-byte aligned -- measured: illegal instruction),
//          so the horizontal taps are moved to the OUTPUT side: B holds the three dx filter columns side by side
//          (N = 3*n_c accumulator columns, P_dx[m] = W[dy][dx] . x[f0+m]) and the epilogue forms
//          out[f0+j] = P_0[j-1] + P_1[j] + P_2[j+1] with warp shuffles (+ a small smem exchange at warp edges).
//          Tiles advance by 120 pixels so that every output has both neighbours inside the same 128-row tile.
// Warp roles per CTA (192 threads): warp 0 = TMA producer, warp 1 = TMEM alloc + MMA issuer, warps 2-5 = epilogue.
#include <cuda_bf16.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "common.cuh"
#include "umma.cuh"
#include "umma_ops.cuh"

namespace b200sep {

using bf16 = __nv_bfloat16;
constexpr int kEpiParts = 2;  // epilogue warps per TMEM lane quadrant: the epilogue is latency-bound (0.48 eligible warps per scheduler with 2), so more warps = more overlap
constexpr int kUmmaThreads = 64 + 128 * kEpiParts;  // warp 0 TMA, warp 1 MMA, then 4 * kEpiParts epilogue warps
constexpr int kMaxChannels = 1024;  // per-channel scale/shift staged in shared memory (conv modes)
constexpr int kTileM = 128;
constexpr int kConv3Parts = 2;  // CONV3x3 kernel: epilogue warps per TMEM lane quadrant.  Measured with 4 (16 epilogue warps, 88 registers): 530 us vs 477 us per scale-0 launch under ncu -- the epilogue is not what paces the kernel (profiles/README.md, round 2)
constexpr int kConv3Threads = 64 + 128 * kConv3Parts;
constexpr int kConvStride = 112;  // output pixels per 3x3 tile: TMEM rows 8..119 of the 128 loaded pixels [f0 - 8, f0 + 120), so that loads AND stores start 16-byte aligned

struct UmmaParams {
  int mode;  // 0 GEMM, 1 CONV3x3, 2 UP (ConvTranspose2d k2 s2), 3 DOWN (Conv2d k2 s2), 4 PW (Conv2d 1x1)
  int f_stride, t_mul, t_off;  // implicit-GEMM addressing: tile f0 = blockIdx.x*f_stride, input row = t*t_mul + r + t_off
  int f_off;                   // first input pixel of a tile = f0 + f_off (CONV3x3: -8, so that the 112 outputs of a tile start 16-byte aligned)
  int n_sbuf;                  // CONV3x3: output staging buffers per epilogue half (2 when shared memory allows)
  int b_resident;              // CONV3x3 with one weight tile that fits (Cin = Cout = 48: 83 KB): the whole B operand is loaded ONCE per CTA and the ring carries only A
  uint32_t b_res_off;          //   byte offset of the resident image [num_iters][hi | lo] from the start of dynamic shared memory (after alignment)
  int cluster;                 // conv modes: CTAs per cluster walking tiles of the same weight tile in lockstep; each loads 1/cluster of every B stage and multicasts it
  int n_tile, n_total, tmem_cols;
  int num_iters, ksteps, stages;
  int dbg;  // development switches from env B200SEP_DBG (0 in production): see launch()
  int sleep_ns;  // > 0: waiting producer / epilogue warps sleep between polls (B200SEP_WAIT_SLEEP_NS)
  int num_tiles, n_ftiles, t_tiles;  // persistent tile walk (n_tiles below = tiles along N / output channels)
  uint32_t a_bytes, b_bytes, stage_bytes;
  // CONV
  int n_chunks, kc, T, F, Cin, Cout, n_tiles, n_c;  // n_c = output channels per CTA; n_tile = 3*n_c accumulator columns
  const bf16* wb_hi;
  const bf16* wb_lo;
  // GEMM
  int M, K, rows_per_channel, channels;
  // epilogue
  const float* scale;
  const float* shift;
  int act;  // 0 none, 1 ReLU, 2 GELU (erf)
  bf16* out_hi;
  bf16* out_lo;
  float* out_f32;      // PW only: write plain fp32 instead of a pair
  const bf16* res_hi;  // GEMM / CONV3x3 / PW: residual (output-shaped, own channel count) ADDED after the activation.  UP: skip tensor MULTIPLIED.
  const bf16* res_lo;
  const bf16* mul_hi;  // CONV3x3 / PW: output-shaped tensor multiplied last
  const bf16* mul_lo;
  int out_c_total, out_c_off;  // conv modes: the output occupies channels [out_c_off, out_c_off + Cout) of a (B, out_c_total, T', F') tensor
};


// activation of a whole register group with ONE test of the (kernel-uniform) activation code: inside the unrolled column loops the per-column
// form cost a uniform branch (and, for GELU, an inlined erf with its own selects) per output
template <int N>
__device__ __forceinline__ void act_group(float (&x)[N], int act) {
  if (act == 1) {
#pragma unroll
    for (int j = 0; j < N; ++j) x[j] = fmaxf(x[j], 0.f);
  } else if (act == 2) {
#pragma unroll
    for (int j = 0; j < N; ++j) x[j] = 0.5f * x[j] * (1.f + erff(x[j] * 0.70710678118654752440f));
  }
}

__device__ __forceinline__ void split_store2(float v, bf16& hi, bf16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}

struct TileCoord {
  int m0, n_idx, f0, t, b;
};
// Tile order keeps concurrently running CTAs on neighbouring tiles (same A rows / same weights stay hot in L2).
__device__ __forceinline__ TileCoord decode_tile(const UmmaParams& p, int tile) {
  TileCoord c{0, 0, 0, 0, 0};
  if (p.mode == 0) {
    c.n_idx = tile % p.n_tiles;
    c.m0 = (tile / p.n_tiles) * kTileM;
  } else {
    const int fx = tile % p.n_ftiles;
    int r = tile / p.n_ftiles;
    c.t = r % p.t_tiles;
    r /= p.t_tiles;
    c.n_idx = r % p.n_tiles;
    c.b = r / p.n_tiles;
    c.f0 = fx * p.f_stride;
  }
  return c;
}

// ===== TMA producer (one thread): fills the shared-memory ring, continuous across the tiles of this CTA =====
__device__ __forceinline__ void umma_producer_loop(const CUtensorMap& tmA_hi, const CUtensorMap& tmA_lo, const CUtensorMap& tmB_hi, const CUtensorMap& tmB_lo,
                                                   const UmmaParams& p, uint8_t* smem, uint64_t* full_bar, uint64_t* empty_bar, uint64_t* wres_bar = nullptr) {
  int s = 0;
  uint32_t phase = 0;
  if (p.b_resident) {  // the layer's whole weight operand, once: [iteration][hi | lo] blocks of b_bytes
    ptx::mbar_arrive_expect_tx(wres_bar, 2u * p.b_bytes * (uint32_t)p.num_iters);
    for (int i = 0; i < p.num_iters; ++i) {
      uint8_t* dst = smem + p.b_res_off + (size_t)i * 2 * p.b_bytes;
      ptx::bulk_load_1d(dst, p.wb_hi + (size_t)i * (p.b_bytes / 2), p.b_bytes, wres_bar);
      ptx::bulk_load_1d(dst + p.b_bytes, p.wb_lo + (size_t)i * (p.b_bytes / 2), p.b_bytes, wres_bar);
    }
  }
  for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
    const TileCoord tc = decode_tile(p, tile);
    const int n0 = tc.n_idx * p.n_tile;
    for (int i = 0; i < p.num_iters; ++i) {
      ptx::mbar_wait_opt(&empty_bar[s], phase ^ 1, p.sleep_ns, 100 + i);
      uint8_t* st = smem + (size_t)s * p.stage_bytes;
      uint8_t* a_hi = st;
      uint8_t* a_lo = st + p.a_bytes;
      uint8_t* b_hi = st + 2 * p.a_bytes;
      uint8_t* b_lo = b_hi + p.b_bytes;
      ptx::mbar_arrive_expect_tx(&full_bar[s], ((p.dbg & 8) ? 0 : 2 * p.a_bytes) + (((p.dbg & 16) || p.b_resident) ? 0 : 2 * p.b_bytes));
      if (p.mode == 0) {
        const int k0 = i * 64;
        if (p.cluster > 1) {
          // the CTAs of a cluster sit on the same 128 activation rows (consecutive weight tiles): this one fetches 128/cluster rows for all of them
          // (tmA_* are then the maps with a [64 k][128/cluster rows] box; rows are 128 bytes, so a slice is whole 1024-byte swizzle atoms)
          const uint32_t rows = 128u / (uint32_t)p.cluster, r0 = ptx::cluster_ctarank() * rows;
          const uint16_t mask = (uint16_t)((1u << p.cluster) - 1u);
          ptx::tma_load_2d_multicast(a_hi + r0 * 128u, &tmA_hi, &full_bar[s], k0, tc.m0 + (int)r0, mask);
          ptx::tma_load_2d_multicast(a_lo + r0 * 128u, &tmA_lo, &full_bar[s], k0, tc.m0 + (int)r0, mask);
        } else if (!(p.dbg & 8)) {
          ptx::tma_load_2d(a_hi, &tmA_hi, &full_bar[s], k0, tc.m0);
          ptx::tma_load_2d(a_lo, &tmA_lo, &full_bar[s], k0, tc.m0);
        }
        if (!(p.dbg & 16)) {
          ptx::tma_load_2d(b_hi, &tmB_hi, &full_bar[s], k0, n0);
          ptx::tma_load_2d(b_lo, &tmB_lo, &full_bar[s], k0, n0);
        }
      } else {
        const int r = i / p.n_chunks, chunk = i - r * p.n_chunks;
        const int cf = tc.f0 + p.f_off, ct = tc.t * p.t_mul + r + p.t_off, cc = tc.b * p.Cin + chunk * p.kc;
        const uint32_t box = (uint32_t)p.kc * 128u;
        if (!(p.dbg & 8)) {
          ptx::tma_load_3d(a_hi, &tmA_hi, &full_bar[s], cf, ct, cc);
          ptx::tma_load_3d(a_hi + box, &tmA_hi, &full_bar[s], cf + 64, ct, cc);
          ptx::tma_load_3d(a_lo, &tmA_lo, &full_bar[s], cf, ct, cc);
          ptx::tma_load_3d(a_lo + box, &tmA_lo, &full_bar[s], cf + 64, ct, cc);
        }
        const size_t woff = ((size_t)tc.n_idx * p.num_iters + i) * (size_t)(p.b_bytes / 2);
        if (p.b_resident) {
          // nothing to fetch: the weights are resident
        } else if (p.cluster > 1) {
          // the CTAs of a cluster are at the same (weight tile, iteration): this one fetches its 1/cluster share of the stage for all of them
          const uint32_t slice = p.b_bytes / (uint32_t)p.cluster, off = ptx::cluster_ctarank() * slice;
          const uint16_t mask = (uint16_t)((1u << p.cluster) - 1u);
          ptx::bulk_load_1d_multicast(b_hi + off, p.wb_hi + woff + off / 2, slice, &full_bar[s], mask);
          ptx::bulk_load_1d_multicast(b_lo + off, p.wb_lo + woff + off / 2, slice, &full_bar[s], mask);
        } else if (!(p.dbg & 16)) {
          ptx::bulk_load_1d(b_hi, p.wb_hi + woff, p.b_bytes, &full_bar[s]);
          ptx::bulk_load_1d(b_lo, p.wb_lo + woff, p.b_bytes, &full_bar[s]);
        }
      }
      if (++s == p.stages) {
        s = 0;
        phase ^= 1;
      }
    }
  }
}

// ===== MMA issuer (one thread): three bf16 UMMAs per k-step into one of two TMEM accumulators =====
__device__ __forceinline__ void umma_mma_loop(const UmmaParams& p, uint8_t* smem, uint64_t* full_bar, uint64_t* empty_bar, uint64_t* tmem_full_bar,
                                              uint64_t* tmem_empty_bar, uint32_t tmem_base, uint32_t acc_stride, uint64_t* wres_bar = nullptr) {
  const uint32_t idesc = ptx::instr_desc_bf16(kTileM, p.n_tile, p.mode != 0 ? 1 : 0, 0);
  if (p.b_resident) ptx::mbar_wait(wres_bar, 0, 500);  // the resident weight image has landed
  int s = 0, acc = 0;
  uint32_t phase = 0, acc_phase = 0;
  for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
    ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1, 400 + acc);  // epilogue has drained this accumulator
    ptx::tc_fence_after();
    const uint32_t d_tmem = tmem_base + (uint32_t)acc * acc_stride;
    for (int i = 0; i < p.num_iters; ++i) {
      ptx::mbar_wait(&full_bar[s], phase, 200 + i);
      ptx::tc_fence_after();
      const uint32_t st = ptx::smem_u32(smem + (size_t)s * p.stage_bytes);
      const uint32_t a_hi = st, a_lo = st + p.a_bytes;
      const uint32_t b_hi = p.b_resident ? ptx::smem_u32(smem + p.b_res_off + (size_t)i * 2 * p.b_bytes) : st + 2 * p.a_bytes, b_lo = b_hi + p.b_bytes;
      for (int j = 0; j < ((p.dbg & 4) ? 0 : p.ksteps); ++j) {
        uint64_t dah, dal, dbh, dbl;
        if (p.mode == 0) {
          dah = ptx::smem_desc(a_hi + j * 32, 16, 1024, ptx::kLayoutSW128);
          dal = ptx::smem_desc(a_lo + j * 32, 16, 1024, ptx::kLayoutSW128);
          dbh = ptx::smem_desc(b_hi + j * 32, 16, 1024, ptx::kLayoutSW128);
          dbl = ptx::smem_desc(b_lo + j * 32, 16, 1024, ptx::kLayoutSW128);
        } else {
          const uint32_t lbo = (uint32_t)p.kc * 128u;  // next 64 pixels (second TMA box)
          dah = ptx::smem_desc(a_hi + j * 2048, lbo, 1024, ptx::kLayoutSW128);
          dal = ptx::smem_desc(a_lo + j * 2048, lbo, 1024, ptx::kLayoutSW128);
          const uint32_t bstep = (uint32_t)p.n_tile * 32u;  // one [n_tile][16] block of 8x8 core matrices
          dbh = ptx::smem_desc(b_hi + j * bstep, 128, 256, ptx::kLayoutNone);
          dbl = ptx::smem_desc(b_lo + j * bstep, 128, 256, ptx::kLayoutNone);
        }
        ptx::umma_bf16(d_tmem, dah, dbh, idesc, (i | j) != 0 ? 1u : 0u);
        ptx::umma_bf16(d_tmem, dah, dbl, idesc, 1u);
        ptx::umma_bf16(d_tmem, dal, dbh, idesc, 1u);
      }
      // frees the smem stage once these MMAs have read it -- in every CTA of the cluster when the stage was filled by multicast
      if (p.cluster > 1) ptx::umma_commit_multicast(&empty_bar[s], (uint16_t)((1u << p.cluster) - 1u));
      else ptx::umma_commit(&empty_bar[s]);
      if (++s == p.stages) {
        s = 0;
        phase ^= 1;
      }
    }
    ptx::umma_commit(&tmem_full_bar[acc]);
    acc ^= 1;
    if (acc == 0) acc_phase ^= 1;
  }
}

// Persistent kernel: grid = min(#tiles, #SMs); every CTA walks tiles blockIdx.x, +gridDim.x, ...  Three pipelines run
// concurrently: TMA producer -> smem ring (full/empty mbarriers, continuous across tiles), MMA issuer -> one of two TMEM
// accumulators (tmem_full/tmem_empty), epilogue warps draining the other accumulator.
__global__ void __launch_bounds__(kUmmaThreads, 1) umma_pair_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                                                                    const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
                                                                    const UmmaParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment for SWIZZLE_128B tiles.  The offset is applied to the __shared__ array itself (not through an integer
  // round trip) so every derived pointer keeps the shared address space: LDS/STS instead of generic LD/ST in the epilogue.
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * p.stage_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tmem_full_bar = empty_bar + p.stages;  // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  float* sc_s = reinterpret_cast<float*>(tmem_slot + 4);  // conv modes: folded BatchNorm scale / shift per output channel
  float* sh_s = sc_s + kMaxChannels;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], p.cluster > 1 ? p.cluster : 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full_bar[a], 1);
      ptx::mbar_init(&tmem_empty_bar[a], 4 * kEpiParts);  // one arrive per epilogue warp
    }
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tmA_hi);
    ptx::prefetch_tensormap(&tmA_lo);
    if (p.mode == 0) {
      ptx::prefetch_tensormap(&tmB_hi);
      ptx::prefetch_tensormap(&tmB_lo);
    }
  }
  if (warp == 1) ptx::tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  if (p.mode != 0) {
    for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) {
      sc_s[i] = p.scale ? __ldg(&p.scale[i]) : 1.f;
      sh_s[i] = p.shift ? __ldg(&p.shift[i]) : 0.f;
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (p.cluster > 1) ptx::cluster_sync();  // every CTA's barriers exist before a peer multicasts into them
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t acc_stride = (uint32_t)p.tmem_cols / 2;

  if (warp == 0) {
    if (lane == 0) umma_producer_loop(tmA_hi, tmA_lo, tmB_hi, tmB_lo, p, smem, full_bar, empty_bar);
  } else if (warp == 1) {
    if (lane == 0) umma_mma_loop(p, smem, full_bar, empty_bar, tmem_full_bar, tmem_empty_bar, tmem_base, acc_stride);
  } else {
    // ===== epilogue: TMEM -> registers -> BN/ReLU(/+res, *skip) -> split into bf16 hi/lo -> global =====
    // Eight warps: warp w may only touch TMEM lanes 32*(w%4)..+31, so two warps share each lane quadrant and split
    // the accumulator columns between them (two warps per scheduler also hide the ALU latency of the conversion chain).
    const int q = warp & 3;
    const int half = (warp - 2) >> 2;
    const int m = q * 32 + lane;
    const int ncol = (p.mode == 0) ? p.n_tile : p.n_c;  // columns of ONE logical output group
    // GEMM: 16-column groups; conv modes: 8-column groups (n_c = 48 splits 24/24 between the two warps of a quadrant)
    const int cw = (p.mode == 0) ? 16 : 8;
    const int nchunks = ncol / cw;
    const int ch_begin = half * nchunks / kEpiParts, ch_end = (half + 1) * nchunks / kEpiParts;  // `half` = which of the kEpiParts column parts
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      const TileCoord tc = decode_tile(p, tile);
      const int m0 = tc.m0, f0 = tc.f0, t = tc.t, b = tc.b;
      const int n0 = tc.n_idx * ncol;
      // GEMM: the residual does not depend on the accumulator -> fetch it while the MMAs of this tile are still running
      uint4 rh[4][2], rl[4][2];
      if (p.mode == 0 && p.res_hi && !(p.dbg & 1)) {
        const int r = m0 + m;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int n = n0 + (ch_begin + k) * 16;
          if (ch_begin + k < ch_end && r < p.M && n < p.n_total) {
            const size_t o = (size_t)r * p.n_total + n;
            rh[k][0] = __ldg(reinterpret_cast<const uint4*>(p.res_hi + o));
            rh[k][1] = __ldg(reinterpret_cast<const uint4*>(p.res_hi + o) + 1);
            rl[k][0] = __ldg(reinterpret_cast<const uint4*>(p.res_lo + o));
            rl[k][1] = __ldg(reinterpret_cast<const uint4*>(p.res_lo + o) + 1);
          }
        }
      }
      ptx::mbar_wait_opt(&tmem_full_bar[acc], acc_phase, p.sleep_ns, 300 + acc);
      ptx::tc_fence_after();
      const uint32_t trow = tmem_base + (uint32_t)acc * acc_stride + ((uint32_t)(q * 32) << 16);
      if (p.dbg & 32) {
        // development: handshake only
      } else if (p.mode == 0) {
        const int r = m0 + m;
        float sc = 1.f, sh = 0.f;
        if (r < p.M) {
          const int c = (r / p.rows_per_channel) % p.channels;
          sc = p.scale ? __ldg(&p.scale[c]) : 1.f;
          sh = p.shift ? __ldg(&p.shift[c]) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int ch = ch_begin + k;
          if (ch >= ch_end) break;
          const int c0 = ch * 16;
          uint32_t v[16];
          ptx::tmem_ld16(trow + (uint32_t)c0, v);
          ptx::tmem_ld_wait();
          const int n = n0 + c0;
          if (r < p.M && n < p.n_total) {
            const size_t o = (size_t)r * p.n_total + n;
            float x[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) x[j] = fmaf(__uint_as_float(v[j]), sc, sh);
            act_group(x, p.act);
            if (p.res_hi && !(p.dbg & 1)) {
              const bf16* h = reinterpret_cast<const bf16*>(rh[k]);
              const bf16* l = reinterpret_cast<const bf16*>(rl[k]);
#pragma unroll
              for (int j = 0; j < 16; ++j) x[j] += __bfloat162float(h[j]) + __bfloat162float(l[j]);
            }
            __align__(16) bf16 oh[16];
            __align__(16) bf16 ol[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) split_store2(x[j], oh[j], ol[j]);
            uint4* dh = reinterpret_cast<uint4*>(p.out_hi + o);
            uint4* dl = reinterpret_cast<uint4*>(p.out_lo + o);
            dh[0] = reinterpret_cast<const uint4*>(oh)[0];
            dh[1] = reinterpret_cast<const uint4*>(oh)[1];
            dl[0] = reinterpret_cast<const uint4*>(ol)[0];
            dl[1] = reinterpret_cast<const uint4*>(ol)[1];
          }
        }
      } else if (p.mode == 2) {
        // ConvTranspose2d k2 s2: column (dy*2+dx)*n_c + co of lane m is the output pixel (2t+dy, 2(f0+m)+dx) of channel co;
        // then BN + ReLU, times the skip tensor (uvr_lib_v5/mdxnet.py:111-112).  The two dx values are stored as one 4-byte pair.
        constexpr int CW = 8;
        const int nc = p.n_c;
        const int f = f0 + m;
        const bool row_ok = f < p.F;
        const int T2 = 2 * p.T, F2 = 2 * p.F;
        const size_t plane = (size_t)T2 * F2;
        for (int dy = 0; dy < 2; ++dy) {
          const size_t base = ((size_t)b * p.out_c_total + p.out_c_off + n0) * plane + (size_t)(2 * t + dy) * F2 + 2 * f;
          const size_t sbase = ((size_t)b * p.Cout + n0) * plane + (size_t)(2 * t + dy) * F2 + 2 * f;  // skip tensor: own channel count
          for (int ch = ch_begin; ch < ch_end; ++ch) {
            const int c0 = ch * CW;
            uint32_t v0[CW], v1[CW];
            ptx::tmem_ld8(trow + (uint32_t)((dy * 2 + 0) * nc + c0), v0);
            ptx::tmem_ld8(trow + (uint32_t)((dy * 2 + 1) * nc + c0), v1);
            ptx::tmem_ld_wait();
            if (row_ok) {
              const size_t o0 = base + (size_t)c0 * plane, s0 = sbase + (size_t)c0 * plane;
              // all skip loads of this group are issued before any store (read-only path)
              uint32_t sk_h[CW], sk_l[CW];
#pragma unroll
              for (int j = 0; j < CW; ++j) {
                sk_h[j] = 0x3f803f80u;  // bf16 (1.0, 1.0)
                sk_l[j] = 0u;
                if (p.res_hi && !(p.dbg & 1)) {
                  sk_h[j] = __ldg(reinterpret_cast<const unsigned int*>(p.res_hi + s0 + (size_t)j * plane));
                  sk_l[j] = __ldg(reinterpret_cast<const unsigned int*>(p.res_lo + s0 + (size_t)j * plane));
                }
              }
              float scv[CW], shv[CW];
#pragma unroll
              for (int j4 = 0; j4 < CW / 4; ++j4) {
                const float4 s4 = *reinterpret_cast<const float4*>(&sc_s[n0 + c0 + 4 * j4]);
                const float4 h4 = *reinterpret_cast<const float4*>(&sh_s[n0 + c0 + 4 * j4]);
                scv[4 * j4] = s4.x; scv[4 * j4 + 1] = s4.y; scv[4 * j4 + 2] = s4.z; scv[4 * j4 + 3] = s4.w;
                shv[4 * j4] = h4.x; shv[4 * j4 + 1] = h4.y; shv[4 * j4 + 2] = h4.z; shv[4 * j4 + 3] = h4.w;
              }
              bf16* ph = p.out_hi + o0;
              bf16* pl = p.out_lo + o0;
              float xa[CW], xb[CW];
#pragma unroll
              for (int j = 0; j < CW; ++j) {
                xa[j] = fmaf(__uint_as_float(v0[j]), scv[j], shv[j]);
                xb[j] = fmaf(__uint_as_float(v1[j]), scv[j], shv[j]);
              }
              act_group(xa, p.act);
              act_group(xb, p.act);
#pragma unroll
              for (int j = 0; j < CW; ++j) {
                // bf16 -> fp32 is a 16-bit shift: low half = element 0 (dx = 0), high half = element 1 (dx = 1)
                float x0 = xa[j] * (__uint_as_float(sk_h[j] << 16) + __uint_as_float(sk_l[j] << 16));
                float x1 = xb[j] * (__uint_as_float(sk_h[j] & 0xffff0000u) + __uint_as_float(sk_l[j] & 0xffff0000u));
                __nv_bfloat162 oh, ol;
                split_store2(x0, oh.x, ol.x);
                split_store2(x1, oh.y, ol.y);
                *reinterpret_cast<__nv_bfloat162*>(ph) = oh;  // 32 lanes -> 128 contiguous bytes
                *reinterpret_cast<__nv_bfloat162*>(pl) = ol;
                ph += plane;
                pl += plane;
              }
            }
          }
        }
      } else if (p.mode == 3) {
        // Conv2d k2 s2: P_dx[m] (column dx*n_c + co) is the partial sum over (ci, dy) at INPUT pixel f0+m;
        // out[(f0+m)/2] = P_0[m] + P_1[m+1] for even m (odd rows of P_0 / even rows of P_1 are computed but unused).
        constexpr int CW = 8;
        const int nc = p.n_c;
        const int fo = (f0 + m) >> 1, Fo = p.F >> 1, To = p.T >> 1;
        const bool row_ok = ((m & 1) == 0) && fo < Fo;
        const size_t plane = (size_t)To * Fo;
        const size_t base = ((size_t)b * p.out_c_total + p.out_c_off + n0) * plane + (size_t)t * Fo + fo;
        for (int ch = ch_begin; ch < ch_end; ++ch) {
          const int c0 = ch * CW;
          uint32_t v0[CW], v1[CW];
          ptx::tmem_ld8(trow + (uint32_t)c0, v0);
          ptx::tmem_ld8(trow + (uint32_t)(nc + c0), v1);
          ptx::tmem_ld_wait();
          float x[CW];
#pragma unroll
          for (int j = 0; j < CW; ++j) x[j] = __uint_as_float(v0[j]) + __shfl_down_sync(0xffffffffu, __uint_as_float(v1[j]), 1);  // + P_1 of row m+1
          float sc[CW], sh[CW];
#pragma unroll
          for (int j4 = 0; j4 < CW / 4; ++j4) {
            const float4 s4 = *reinterpret_cast<const float4*>(&sc_s[n0 + c0 + 4 * j4]);
            const float4 h4 = *reinterpret_cast<const float4*>(&sh_s[n0 + c0 + 4 * j4]);
            sc[4 * j4] = s4.x; sc[4 * j4 + 1] = s4.y; sc[4 * j4 + 2] = s4.z; sc[4 * j4 + 3] = s4.w;
            sh[4 * j4] = h4.x; sh[4 * j4 + 1] = h4.y; sh[4 * j4 + 2] = h4.z; sh[4 * j4 + 3] = h4.w;
          }
          if (row_ok) {
            bf16* ph = p.out_hi + base + (size_t)c0 * plane;
            bf16* pl = p.out_lo + base + (size_t)c0 * plane;
            float y[CW];
#pragma unroll
            for (int j = 0; j < CW; ++j) y[j] = fmaf(x[j], sc[j], sh[j]);
            act_group(y, p.act);
#pragma unroll
            for (int j = 0; j < CW; ++j) {
              bf16 h, l;
              split_store2(y[j], h, l);
              *ph = h;
              *pl = l;
              ph += plane;
              pl += plane;
            }
          }
        }
      } else if (p.mode == 4) {
        // 1x1 convolution: column co of lane m is output pixel f0+m of channel n0+co.
        constexpr int CW = 8;
        const int f = f0 + m;
        const bool row_ok = f < p.F;
        const size_t plane = (size_t)p.T * p.F;
        const size_t base = ((size_t)b * p.out_c_total + p.out_c_off + n0) * plane + (size_t)t * p.F + f;
        const size_t rbase = ((size_t)b * p.Cout + n0) * plane + (size_t)t * p.F + f;
        for (int ch = ch_begin; ch < ch_end; ++ch) {
          const int c0 = ch * CW;
          uint32_t v[CW];
          ptx::tmem_ld8(trow + (uint32_t)c0, v);
          ptx::tmem_ld_wait();
          float sc[CW], sh[CW];
#pragma unroll
          for (int j4 = 0; j4 < CW / 4; ++j4) {
            const float4 s4 = *reinterpret_cast<const float4*>(&sc_s[n0 + c0 + 4 * j4]);
            const float4 h4 = *reinterpret_cast<const float4*>(&sh_s[n0 + c0 + 4 * j4]);
            sc[4 * j4] = s4.x; sc[4 * j4 + 1] = s4.y; sc[4 * j4 + 2] = s4.z; sc[4 * j4 + 3] = s4.w;
            sh[4 * j4] = h4.x; sh[4 * j4 + 1] = h4.y; sh[4 * j4 + 2] = h4.z; sh[4 * j4 + 3] = h4.w;
          }
          if (row_ok) {
            float y[CW];
#pragma unroll
            for (int j = 0; j < CW; ++j) y[j] = fmaf(__uint_as_float(v[j]), sc[j], sh[j]);
            act_group(y, p.act);
            if (p.res_hi) {
#pragma unroll
              for (int j = 0; j < CW; ++j) {
                const size_t ro = rbase + (size_t)(c0 + j) * plane;
                y[j] += __bfloat162float(p.res_hi[ro]) + __bfloat162float(p.res_lo[ro]);
              }
            }
            if (p.mul_hi) {
#pragma unroll
              for (int j = 0; j < CW; ++j) {
                const size_t ro = rbase + (size_t)(c0 + j) * plane;
                y[j] *= __bfloat162float(p.mul_hi[ro]) + __bfloat162float(p.mul_lo[ro]);
              }
            }
            if (p.out_f32) {
#pragma unroll
              for (int j = 0; j < CW; ++j) p.out_f32[base + (size_t)(c0 + j) * plane] = y[j];
            } else {
#pragma unroll
              for (int j = 0; j < CW; ++j) {
                const size_t o = base + (size_t)(c0 + j) * plane;
                bf16 h, l;
                split_store2(y[j], h, l);
                p.out_hi[o] = h;
                p.out_lo[o] = l;
              }
            }
          }
        }
      }  // (CONV3x3 has its own kernel, umma_conv3_kernel)
      // this warp is done reading the accumulator: hand it back to the MMA issuer
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (p.cluster > 1) ptx::cluster_sync();  // no CTA leaves while a peer may still signal its barriers
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------
// CONV3x3 kernel.  Same producer / MMA pipelines as umma_pair_kernel; the epilogue is specialised (NC = output channels per CTA):
//   * a tile loads the 128 pixels [f0 - 8, f0 + 120) (TMA zero-fills the left / right padding) and produces the 112 outputs
//     [f0, f0 + 112) = TMEM rows 8..119, so both the loads and the STORES start 16-byte aligned (TMA faults on any other
//     innermost coordinate, measured: tests/dev/tma_probe2.cu);
//   * each of the 8 epilogue warps pulls ALL its accumulator columns (3 * NC/2) into registers with one tcgen05.wait::ld and
//     hands the accumulator back to the MMA issuer at once -- the arithmetic below overlaps the next tiles' MMAs;
//   * out[j] = P_0[j-1] + P_1[j] + P_2[j+1] by warp shuffles, the three warp-boundary rows through a 128-thread exchange
//     (no second pass over TMEM), folded BatchNorm + activation (+ residual, * multiplier), bf16 hi/lo split;
//   * the tile is staged in shared memory as [channel][pixel] bf16 planes and written with two cp.async.bulk.tensor stores per half
//     (UTMASTG): no per-thread global stores, no 64-bit address arithmetic, full 224-byte rows per channel.
template <int NC>
__global__ void __launch_bounds__(kConv3Threads, 1) umma_conv3_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
                                                                     const __grid_constant__ CUtensorMap tmO_hi, const __grid_constant__ CUtensorMap tmO_lo,
                                                                     const UmmaParams p) {
  constexpr int H = NC / kConv3Parts;       // channels per epilogue warp
  constexpr int kPlane = H * kConvStride;   // bf16 elements of one staged plane [H][112]
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  // [ring: stages x stage_bytes][resident weights, when b_resident][output staging][barriers, BN coefficients, edge rows]
  bf16* stage_out = reinterpret_cast<bf16*>(smem + (size_t)p.stages * p.stage_bytes + (p.b_resident ? (size_t)2 * p.b_bytes * p.num_iters : 0));  // [n_sbuf][parts][hi, lo][H][112]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(stage_out) + (size_t)p.n_sbuf * 2 * kConv3Parts * kPlane * sizeof(bf16));
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tmem_full_bar = empty_bar + p.stages;  // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;    // [2]
  uint64_t* wres_bar = tmem_empty_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wres_bar + 2);  // (+2: keeps everything behind it 16-byte aligned -- sc_s / sh_s / the edge rows are read as float4)
  float* sc_s = reinterpret_cast<float*>(tmem_slot + 4);
  float* sh_s = sc_s + kMaxChannels;
  float* edge_base = sh_s + kMaxChannels;  // [kConv3Parts][P_0 row 31 | P_2 row 0][4 quadrants][H]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], p.cluster > 1 ? p.cluster : 1);
    }
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(&tmem_full_bar[a], 1);
      ptx::mbar_init(&tmem_empty_bar[a], 4 * kConv3Parts);
    }
    ptx::mbar_init(wres_bar, 1);
    ptx::fence_barrier_init();
    ptx::prefetch_tensormap(&tmA_hi);
    ptx::prefetch_tensormap(&tmA_lo);
    ptx::prefetch_tensormap(&tmO_hi);
    ptx::prefetch_tensormap(&tmO_lo);
  }
  if (warp == 1) ptx::tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  for (int i = threadIdx.x; i < p.Cout; i += blockDim.x) {
    sc_s[i] = p.scale ? __ldg(&p.scale[i]) : 1.f;
    sh_s[i] = p.shift ? __ldg(&p.shift[i]) : 0.f;
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (p.cluster > 1) ptx::cluster_sync();  // every CTA's barriers exist before a peer multicasts into them
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t acc_stride = (uint32_t)p.tmem_cols / 2;

  if (warp == 0) {
    if (lane == 0) umma_producer_loop(tmA_hi, tmA_lo, tmA_hi, tmA_lo, p, smem, full_bar, empty_bar, wres_bar);
  } else if (warp == 1) {
    if (lane == 0) umma_mma_loop(p, smem, full_bar, empty_bar, tmem_full_bar, tmem_empty_bar, tmem_base, acc_stride, wres_bar);
  } else {
    const int q = warp & 3;           // TMEM lane quadrant
    const int half = (warp - 2) >> 2;  // which NC/kConv3Parts channels
    const int m = q * 32 + lane;
    const bool issuer = (q == 0) && (lane == 0);  // the thread of this half that owns the bulk store groups
    const bool out_row = (m >= 8) && (m < 8 + kConvStride);
    float* edge0 = edge_base + half * 8 * H;  // [q][H]: P_0 of row 32q+31
    float* edge2 = edge0 + 4 * H;             // [q][H]: P_2 of row 32q
    const int bar_a = 1 + 2 * half, bar_b = 2 + 2 * half;
    int acc = 0, it = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
      const TileCoord tc = decode_tile(p, tile);
      const int n0 = tc.n_idx * NC + half * H;  // first output channel of this warp
      ptx::mbar_wait_opt(&tmem_full_bar[acc], acc_phase, p.sleep_ns, 300 + acc);
      ptx::tc_fence_after();
      const uint32_t trow = tmem_base + (uint32_t)acc * acc_stride + ((uint32_t)(q * 32) << 16) + (uint32_t)(half * H);
      uint32_t v0[H], v1[H], v2[H];
      ptx::tmem_ld_n<H>(trow, v0);
      ptx::tmem_ld_n<H>(trow + NC, v1);
      ptx::tmem_ld_n<H>(trow + 2 * NC, v2);
      ptx::tmem_ld_wait();
      // the accumulator now lives in registers: hand it back to the MMA issuer
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&tmem_empty_bar[acc]);
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
      // boundary rows for the neighbouring quadrants
      if (lane == 31) {
#pragma unroll
        for (int j = 0; j < H; j += 4) *reinterpret_cast<uint4*>(&edge0[q * H + j]) = make_uint4(v0[j], v0[j + 1], v0[j + 2], v0[j + 3]);
      }
      if (lane == 0) {
#pragma unroll
        for (int j = 0; j < H; j += 4) *reinterpret_cast<uint4*>(&edge2[q * H + j]) = make_uint4(v2[j], v2[j + 1], v2[j + 2], v2[j + 3]);
      }
      // the staging buffer of this tile must have been read out by the store issued n_sbuf tiles ago
      if (issuer) {
        if (p.n_sbuf == 2) ptx::bulk_wait_read<1>();
        else ptx::bulk_wait_read<0>();
      }
      asm volatile("bar.sync %0, 128;" ::"r"(bar_a) : "memory");
      float x[H];
#pragma unroll
      for (int j = 0; j < H; ++j) {
        const float a = __shfl_up_sync(0xffffffffu, __uint_as_float(v0[j]), 1);    // P_0 of row m-1
        const float c = __shfl_down_sync(0xffffffffu, __uint_as_float(v2[j]), 1);  // P_2 of row m+1
        x[j] = __uint_as_float(v1[j]) + ((lane == 0) ? 0.f : a) + ((lane == 31) ? 0.f : c);
      }
      if (lane == 0 && q > 0) {
#pragma unroll
        for (int j = 0; j < H; j += 4) {
          const float4 e = *reinterpret_cast<const float4*>(&edge0[(q - 1) * H + j]);
          x[j] += e.x; x[j + 1] += e.y; x[j + 2] += e.z; x[j + 3] += e.w;
        }
      }
      if (lane == 31 && q < 3) {
#pragma unroll
        for (int j = 0; j < H; j += 4) {
          const float4 e = *reinterpret_cast<const float4*>(&edge2[(q + 1) * H + j]);
          x[j] += e.x; x[j + 1] += e.y; x[j + 2] += e.z; x[j + 3] += e.w;
        }
      }
#pragma unroll
      for (int j = 0; j < H; j += 4) {
        const float4 s4 = *reinterpret_cast<const float4*>(&sc_s[n0 + j]);
        const float4 h4 = *reinterpret_cast<const float4*>(&sh_s[n0 + j]);
        x[j] = fmaf(x[j], s4.x, h4.x); x[j + 1] = fmaf(x[j + 1], s4.y, h4.y); x[j + 2] = fmaf(x[j + 2], s4.z, h4.z); x[j + 3] = fmaf(x[j + 3], s4.w, h4.w);
      }
      act_group(x, p.act);
      const int f = tc.f0 + m - 8;
      if ((p.res_hi || p.mul_hi) && out_row && f < p.F) {
        const size_t plane = (size_t)p.T * p.F;
        const size_t rbase = ((size_t)tc.b * p.Cout + n0) * plane + (size_t)tc.t * p.F + f;  // residual / multiplier: (B, Cout, T, F)
        if (p.res_hi) {
#pragma unroll
          for (int j = 0; j < H; ++j) x[j] += __bfloat162float(p.res_hi[rbase + (size_t)j * plane]) + __bfloat162float(p.res_lo[rbase + (size_t)j * plane]);
        }
        if (p.mul_hi) {
#pragma unroll
          for (int j = 0; j < H; ++j) x[j] *= __bfloat162float(p.mul_hi[rbase + (size_t)j * plane]) + __bfloat162float(p.mul_lo[rbase + (size_t)j * plane]);
        }
      }
      bf16* s_hi = stage_out + (size_t)(((p.n_sbuf == 2) ? (it & 1) : 0) * kConv3Parts + half) * 2 * kPlane;
      bf16* s_lo = s_hi + kPlane;
      if (out_row) {
#pragma unroll
        for (int j = 0; j < H; ++j) {
          bf16 h, l;
          split_store2(x[j], h, l);
          s_hi[j * kConvStride + (m - 8)] = h;
          s_lo[j * kConvStride + (m - 8)] = l;
        }
      }
      ptx::fence_proxy_async();
      asm volatile("bar.sync %0, 128;" ::"r"(bar_b) : "memory");
      if (issuer) {
        const int cc = tc.b * p.out_c_total + p.out_c_off + n0;
        ptx::tma_store_3d(&tmO_hi, s_hi, tc.f0, tc.t, cc);
        ptx::tma_store_3d(&tmO_lo, s_lo, tc.f0, tc.t, cc);
        ptx::bulk_commit();
      }
    }
    if (issuer) ptx::bulk_wait_all();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (p.cluster > 1) ptx::cluster_sync();  // no CTA leaves while a peer may still signal its barriers
  if (warp == 1) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------
// host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                    const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// bf16 tensor map, SWIZZLE_128B, zero OOB fill.  dims/box innermost first; strides in BYTES for dims 1..rank-1.
static int make_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes, const uint32_t* box,
                    CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return B200SEP_ERR_CUDA;
  }
  cuuint64_t gd[5], gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) gs[i - 1] = strides_bytes[i - 1];
  }
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (CUresult %d) rank=%d dims=[%llu,%llu,%llu] box=[%u,%u,%u]", (int)r, rank, (unsigned long long)dims[0],
              (unsigned long long)(rank > 1 ? dims[1] : 0), (unsigned long long)(rank > 2 ? dims[2] : 0), box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0);
    return B200SEP_ERR_CUDA;
  }
  return B200SEP_OK;
}

static int pow2_cols(int n) {
  int c = 32;
  while (c < n) c <<= 1;
  return c;
}

static int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = kNumSMs;
  }
  return n;
}

// Cluster size for the operand multicast.  Conv modes: the CTAs of a cluster must sit on the same weight tile at every step of their tile walk, which holds
// when tile ids, the grid and the number of tiles per weight tile are all multiples of the cluster size; GEMM: `cs` consecutive tiles share their activation rows
// when cs divides the tiles along N.  Measured on B200 (profiles/README.md, round 2): the conv kernels gain nothing from it (they are not L2-bound), so it is
// off by default there; B200SEP_CLUSTER / B200SEP_CLUSTER_GEMM (1, 2, 4, 8) select it for A/B runs.
static int env_cluster(const char* name, int dflt) {
  const char* e = getenv(name);
  const int v = e ? atoi(e) : dflt;
  return (v == 1 || v == 2 || v == 4 || v == 8) ? v : dflt;
}
static int umma_wait_sleep_ns() {
  static const int ns = [] {
    const char* e = getenv("B200SEP_WAIT_SLEEP_NS");
    return e ? atoi(e) : 0;
  }();
  return ns;
}

static int choose_cluster(const UmmaParams& p) {
  static const int want_conv = env_cluster("B200SEP_CLUSTER", 1), want_gemm = env_cluster("B200SEP_CLUSTER_GEMM", 1);
  if (p.mode == 0) {
    for (int cs = std::min(want_gemm, 4); cs > 1; cs >>= 1)
      if (p.n_tiles % cs == 0) return cs;
    return 1;
  }
  for (int cs = want_conv; cs > 1; cs >>= 1)
    if (p.num_tiles % cs == 0 && (p.n_ftiles * p.t_tiles) % cs == 0 && p.b_bytes % (16u * cs) == 0) return cs;
  return 1;
}

// Persistent launch: one CTA per SM, as clusters of `cs` when the weight operand is multicast (the grid is then the number of co-resident clusters x cs).
template <class Kernel, class... Args>
static int launch_persistent(Kernel kernel, int threads, int cs, int num_tiles, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int grid = std::min(num_tiles, num_sms());
  if (cs > 1) {
    static std::map<std::tuple<const void*, int, size_t>, int> cache;
    static std::mutex mu;
    int nclusters = 0;
    {
      std::lock_guard<std::mutex> lock(mu);
      const auto key = std::make_tuple((const void*)kernel, cs, smem);
      auto it = cache.find(key);
      if (it == cache.end()) {
        cfg.gridDim = dim3((unsigned)(num_sms() / cs * cs));
        B2_CUDA(cudaOccupancyMaxActiveClusters(&nclusters, kernel, &cfg));
        cache[key] = nclusters;
      } else {
        nclusters = it->second;
      }
    }
    B2_CHECK_ARG(nclusters >= 1, "umma: no cluster of %d CTAs with %zu bytes of shared memory can be resident", cs, smem);
    grid = std::min(num_tiles, nclusters * cs) / cs * cs;
  }
  cfg.gridDim = dim3((unsigned)grid);
  B2_CUDA(cudaLaunchKernelEx(&cfg, kernel, args...));
  count_launch();
  return B200SEP_OK;
}

// `tiles` is the logical tile grid: GEMM (n tiles, m tiles, 1); conv modes (f tiles, output rows, batch * channel tiles).
static int launch(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi, const CUtensorMap& b_lo, UmmaParams& p, dim3 tiles,
                  cudaStream_t st, const CUtensorMap* a_slices = nullptr /* GEMM: {hi, lo} with 64-row boxes, {hi, lo} with 32-row boxes */) {
  {
    const char* e = getenv("B200SEP_DBG");  // development only: selectively disable parts of the kernel (results become wrong)
    p.dbg = e ? atoi(e) : 0;
    p.sleep_ns = umma_wait_sleep_ns();
  }
  p.stage_bytes = ((2 * p.a_bytes + 2 * p.b_bytes + 1023) / 1024) * 1024;
  p.tmem_cols = 2 * pow2_cols(p.n_tile);  // two accumulators: the epilogue of tile i overlaps the MMAs of tile i+1
  B2_CHECK_ARG(p.tmem_cols <= 512, "umma: n_tile=%d needs more than 512 TMEM columns", p.n_tile);
  if (p.mode == 0) p.n_tiles = (int)tiles.x;
  p.n_ftiles = (int)tiles.x;
  p.t_tiles = (int)tiles.y;
  p.num_tiles = (int)(tiles.x * tiles.y * tiles.z);
  const size_t fixed = 1024 /*alignment slack*/ + 64 * sizeof(uint64_t) + 64 + 2 * kMaxChannels * sizeof(float) + (p.mode != 0 ? (size_t)16 * p.n_c * sizeof(float) : 0);
  B2_CHECK_ARG(p.mode == 0 || p.Cout <= kMaxChannels, "umma: more than %d output channels", kMaxChannels);
  const size_t budget = 220 * 1024 - fixed;  // one persistent CTA per SM
  int stages = (int)(budget / p.stage_bytes);
  if (stages > 8) stages = 8;
  B2_CHECK_ARG(stages >= 2, "umma: a pipeline stage of %u bytes does not fit twice in shared memory", p.stage_bytes);
  p.stages = stages;
  const size_t smem = (size_t)stages * p.stage_bytes + fixed;
  static bool attr_set = false;
  if (!attr_set) {
    B2_CUDA(cudaFuncSetAttribute(umma_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  p.cluster = choose_cluster(p);
  if (p.mode == 0 && p.cluster > 1) {
    B2_CHECK_ARG(a_slices != nullptr, "umma: GEMM multicast needs the sliced activation maps");
    const CUtensorMap* sl = a_slices + (p.cluster == 4 ? 2 : 0);
    return launch_persistent(umma_pair_kernel, kUmmaThreads, p.cluster, p.num_tiles, smem, st, sl[0], sl[1], b_hi, b_lo, p);
  }
  return launch_persistent(umma_pair_kernel, kUmmaThreads, p.cluster, p.num_tiles, smem, st, a_hi, a_lo, b_hi, b_lo, p);
}

bool umma_gemm_supported(int M, int N, int K) { return M >= 1 && N % 16 == 0 && K % 8 == 0 && N >= 16 && K >= 16; }

int umma_gemm_plan_create(UmmaGemmPlan* pl, const void* a_hi, const void* a_lo, const void* w_hi, const void* w_lo, int M, int N, int K) {
  pl->M = M; pl->N = N; pl->K = K;
  int n_tile = N <= 128 ? N : 128;
  if (N > 128 && N % 128 != 0) {
    for (n_tile = 128; n_tile >= 16; n_tile -= 16)
      if (N % n_tile == 0) break;
  }
  // prefer a tile width whose tile count along N is a multiple of 4 (then of 2): those tiles run as one cluster and share the activation rows by multicast
  auto share = [&](int nt) { const int t = N / nt; return t % 4 == 0 ? 4 : (t % 2 == 0 ? 2 : 1); };
  for (int cand : {96, 64})
    if (N % cand == 0 && N >= cand && share(cand) > share(n_tile)) n_tile = cand;
  pl->n_tile = n_tile;
  const uint64_t da[2] = {(uint64_t)K, (uint64_t)M}, sa[1] = {(uint64_t)K * 2};
  const uint32_t ba[2] = {64, 128};
  const uint64_t db[2] = {(uint64_t)K, (uint64_t)N};
  const uint32_t bb[2] = {64, (uint32_t)n_tile};
  int rc = make_map(&pl->a_hi, a_hi, 2, da, sa, ba);
  if (!rc) rc = make_map(&pl->a_lo, a_lo, 2, da, sa, ba);
  const uint32_t ba2[2] = {64, 64}, ba4[2] = {64, 32};
  if (!rc) rc = make_map(&pl->a_slices[0], a_hi, 2, da, sa, ba2);
  if (!rc) rc = make_map(&pl->a_slices[1], a_lo, 2, da, sa, ba2);
  if (!rc) rc = make_map(&pl->a_slices[2], a_hi, 2, da, sa, ba4);
  if (!rc) rc = make_map(&pl->a_slices[3], a_lo, 2, da, sa, ba4);
  if (!rc) rc = make_map(&pl->b_hi, w_hi, 2, db, sa, bb);
  if (!rc) rc = make_map(&pl->b_lo, w_lo, 2, db, sa, bb);
  return rc;
}

static void fill_epilogue(UmmaParams& p, const UmmaEpilogue& e, int Cout) {
  p.scale = e.scale; p.shift = e.shift; p.act = e.act;
  p.out_hi = (bf16*)e.out_hi; p.out_lo = (bf16*)e.out_lo; p.out_f32 = e.out_f32;
  p.res_hi = (const bf16*)e.res_hi; p.res_lo = (const bf16*)e.res_lo;
  p.mul_hi = (const bf16*)e.mul_hi; p.mul_lo = (const bf16*)e.mul_lo;
  p.out_c_total = e.out_c_total > 0 ? e.out_c_total : Cout;
  p.out_c_off = e.out_c_off;
}

int umma_gemm_run(const UmmaGemmPlan& pl, const float* scale, const float* shift, int rows_per_channel, int channels, int relu, void* out_hi,
                  void* out_lo, const void* res_hi, const void* res_lo, int M_active, cudaStream_t st) {
  UmmaEpilogue e;
  e.scale = scale; e.shift = shift; e.act = relu ? 1 : 0; e.out_hi = out_hi; e.out_lo = out_lo; e.res_hi = res_hi; e.res_lo = res_lo;
  return umma_gemm_run_ex(pl, rows_per_channel, channels, M_active, e, st);
}

int umma_gemm_run_ex(const UmmaGemmPlan& pl, int rows_per_channel, int channels, int M_active, const UmmaEpilogue& e, cudaStream_t st) {
  const float* scale = e.scale; const float* shift = e.shift; const int relu = e.act;
  void* out_hi = e.out_hi; void* out_lo = e.out_lo; const void* res_hi = e.res_hi; const void* res_lo = e.res_lo;
  UmmaParams p{};
  p.mode = 0;
  p.n_tile = pl.n_tile; p.n_total = pl.N;
  p.num_iters = (pl.K + 63) / 64; p.ksteps = 4;
  p.a_bytes = 128 * 128; p.b_bytes = (uint32_t)pl.n_tile * 128;
  p.M = M_active; p.K = pl.K; p.rows_per_channel = rows_per_channel; p.channels = channels;
  p.scale = scale; p.shift = shift; p.act = relu;
  p.out_hi = (bf16*)out_hi; p.out_lo = (bf16*)out_lo; p.res_hi = (const bf16*)res_hi; p.res_lo = (const bf16*)res_lo;
  B2_CHECK_ARG(pl.n_tile <= 128, "umma_gemm: n_tile=%d exceeds the epilogue's 8 column groups", pl.n_tile);
  dim3 grid(pl.N / pl.n_tile, cdiv(M_active, kTileM));
  return launch(pl.a_hi, pl.a_lo, pl.b_hi, pl.b_lo, p, grid, st, pl.a_slices);
}

bool umma_conv_supported(int Cin, int Cout, int F, int kh, int kw) {
  return Cin % 16 == 0 && Cout % 16 == 0 && F % 8 == 0 && kh == 3 && kw == 3;
}

// kc = input channels per pipeline stage, n_c = output channels per CTA (3*n_c accumulator columns <= 256)
int umma_conv_choose(int Cin, int Cout, int* kc, int* n_c) {
  int k = 64;
  while (k > 16 && Cin % k != 0) k -= 16;
  if (Cin % 48 == 0) k = 48;
  int nc = 16;
  const int cand[5] = {48, 80, 64, 32, 16};
  for (int i = 0; i < 5; ++i)
    if (Cout % cand[i] == 0) {
      nc = cand[i];
      break;
    }
  // the ring needs at least two stages next to the output staging tile of the TMA-store epilogue: shrink the channel step of wide tiles
  // (n_c = 80 with 64 channels per stage is a 92 KB stage: MDX23C's 640-channel scale)
  auto fits = [&](int kk) {
    const size_t stage = ((size_t)2 * kk * 256 + (size_t)2 * (kk / 16) * (3 * nc) * 32 + 1023) / 1024 * 1024;
    const size_t staging = (size_t)2 * kConv3Parts * (nc / kConv3Parts) * kConvStride * 2;
    return 2 * stage + staging + 16 * 1024 <= 227 * 1024;
  };
  while (!fits(k) && k > 16) {
    int kk = k - 16;
    while (kk > 16 && Cin % kk != 0) kk -= 16;
    if (Cin % kk != 0) break;
    k = kk;
  }
  *kc = k;
  *n_c = nc;
  return 0;
}

int umma_conv_plan_create(UmmaConvPlan* pl, const void* x_hi, const void* x_lo, int Bmax, int Cin, int T, int F, int kc) {
  pl->Cin = Cin; pl->T = T; pl->F = F; pl->kc = kc;
  const uint64_t d[3] = {(uint64_t)F, (uint64_t)T, (uint64_t)Bmax * Cin};
  const uint64_t s[2] = {(uint64_t)F * 2, (uint64_t)T * F * 2};
  const uint32_t bx[3] = {64, 1, (uint32_t)kc};
  int rc = make_map(&pl->a_hi, x_hi, 3, d, s, bx);
  if (!rc) rc = make_map(&pl->a_lo, x_lo, 3, d, s, bx);
  return rc;
}

int umma_conv_run(const UmmaConvPlan& pl, const void* wb_hi, const void* wb_lo, int B, int Cout, int n_c, int ksize, const float* scale,
                  const float* shift, int relu, void* out_hi, void* out_lo, cudaStream_t st) {
  B2_CHECK_ARG(ksize == 3, "umma_conv: only 3x3 kernels");
  UmmaEpilogue e;
  e.scale = scale; e.shift = shift; e.act = relu ? 1 : 0; e.out_hi = out_hi; e.out_lo = out_lo;
  return umma_conv_run_ex(pl, wb_hi, wb_lo, B, Cout, n_c, e, st);
}

// TMA store maps of a conv3x3 output: the (F, T, B * C_total) bf16 planes with a [112 px][1 row][NC/2 channels] box, no swizzle.  Encoding a map costs a few
// microseconds on the host and the same activation buffers are written forward after forward, so the maps are cached by (plane address, geometry).
struct StoreMapKey {
  const void* base; int F, T, C, box_c;
  bool operator<(const StoreMapKey& o) const { return std::tie(base, F, T, C, box_c) < std::tie(o.base, o.F, o.T, o.C, o.box_c); }
};
static int store_map(const void* base, int F, int T, int C, int box_c, CUtensorMap* out) {
  static std::map<StoreMapKey, CUtensorMap> cache;
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);
  const StoreMapKey key{base, F, T, C, box_c};
  auto it = cache.find(key);
  if (it == cache.end()) {
    CUtensorMap m;
    const uint64_t d[3] = {(uint64_t)F, (uint64_t)T, (uint64_t)C};
    const uint64_t st[2] = {(uint64_t)F * 2, (uint64_t)T * F * 2};
    const uint32_t bx[3] = {(uint32_t)kConvStride, 1, (uint32_t)box_c};
    int rc = make_map(&m, base, 3, d, st, bx, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    if (cache.size() > 4096) cache.clear();
    it = cache.emplace(key, m).first;
  }
  *out = it->second;
  return B200SEP_OK;
}

template <int NC>
static int launch_conv3(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& o_hi, const CUtensorMap& o_lo, UmmaParams& p, size_t smem, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    B2_CUDA(cudaFuncSetAttribute(umma_conv3_kernel<NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  p.cluster = choose_cluster(p);
  p.sleep_ns = umma_wait_sleep_ns();
  return launch_persistent(umma_conv3_kernel<NC>, kConv3Threads, p.cluster, p.num_tiles, smem, st, a_hi, a_lo, o_hi, o_lo, p);
}

int umma_conv_run_ex(const UmmaConvPlan& pl, const void* wb_hi, const void* wb_lo, int B, int Cout, int n_c, const UmmaEpilogue& e, cudaStream_t st) {
  UmmaParams p{};
  p.mode = 1; p.f_stride = kConvStride; p.f_off = -8; p.t_mul = 1; p.t_off = -1;
  p.n_c = n_c; p.n_tile = 3 * n_c; p.n_total = Cout;
  p.kc = pl.kc; p.n_chunks = pl.Cin / pl.kc;
  p.num_iters = 3 * p.n_chunks; p.ksteps = pl.kc / 16;
  p.a_bytes = (uint32_t)pl.kc * 256; p.b_bytes = (uint32_t)p.ksteps * p.n_tile * 32;
  p.T = pl.T; p.F = pl.F; p.Cin = pl.Cin; p.Cout = Cout; p.n_tiles = Cout / n_c;
  p.wb_hi = (const bf16*)wb_hi; p.wb_lo = (const bf16*)wb_lo;
  fill_epilogue(p, e, Cout);
  B2_CHECK_ARG(Cout <= kMaxChannels, "umma_conv: more than %d output channels", kMaxChannels);
  B2_CHECK_ARG(e.out_f32 == nullptr, "umma_conv: 3x3 convolutions write pair tensors only");
  // one weight tile whose whole B operand fits next to the ring (Cin = Cout = 48: 83 KB): keep it resident; the shared-memory data pipe is the kernel's
  // limiter (TC operand fetch + TMA fill + epilogue stores, profiles/README.md round 2) and the per-tile weight refill was 30 % of the TMA fill
  const size_t b_all = (size_t)2 * p.b_bytes * p.num_iters;
  static const bool allow_res = !(getenv("B200SEP_WRES") && atoi(getenv("B200SEP_WRES")) == 0);
  p.b_resident = (allow_res && p.n_tiles == 1 && b_all <= 96 * 1024) ? 1 : 0;
  p.stage_bytes = ((2 * p.a_bytes + (p.b_resident ? 0 : 2 * p.b_bytes) + 1023) / 1024) * 1024;
  p.tmem_cols = 2 * pow2_cols(p.n_tile);
  B2_CHECK_ARG(p.tmem_cols <= 512, "umma_conv: n_c=%d needs more than 512 TMEM columns", n_c);
  p.n_ftiles = cdiv(pl.F, kConvStride);
  p.t_tiles = pl.T;
  p.num_tiles = p.n_ftiles * pl.T * B * p.n_tiles;
  B2_CHECK_ARG(n_c % (4 * kConv3Parts) == 0, "umma_conv: n_c=%d is not a multiple of %d", n_c, 4 * kConv3Parts);
  const size_t stage_plane = (size_t)(n_c / kConv3Parts) * kConvStride * 2;  // bytes of one staged [n_c/parts][112] bf16 plane
  const size_t fixed = 1024 /*alignment slack*/ + 64 * sizeof(uint64_t) + 64 + 2 * kMaxChannels * sizeof(float) + (size_t)8 * n_c * sizeof(float) +
                       (p.b_resident ? b_all : 0);
  const size_t budget = 227 * 1024 - fixed;
  p.n_sbuf = 2;
  const size_t sbuf_bytes = 2 * kConv3Parts * stage_plane;  // hi + lo plane per column part
  int stages = (int)((budget - 2 * sbuf_bytes) / p.stage_bytes);
  if (stages < 3) {  // deep layers with 80 KB stages: one staging buffer leaves room for the ring
    p.n_sbuf = 1;
    stages = (int)((budget - sbuf_bytes) / p.stage_bytes);
  }
  if (stages > 8) stages = 8;
  B2_CHECK_ARG(stages >= 2, "umma_conv: a pipeline stage of %u bytes does not fit twice in shared memory", p.stage_bytes);
  p.stages = stages;
  p.b_res_off = (uint32_t)((size_t)stages * p.stage_bytes);
  const size_t smem = (size_t)stages * p.stage_bytes + (size_t)p.n_sbuf * sbuf_bytes + fixed;
  CUtensorMap o_hi, o_lo;
  int rc = store_map(p.out_hi, pl.F, pl.T, B * p.out_c_total, n_c / kConv3Parts, &o_hi);
  if (!rc) rc = store_map(p.out_lo, pl.F, pl.T, B * p.out_c_total, n_c / kConv3Parts, &o_lo);
  if (rc) return rc;
  switch (n_c) {
    case 16: return launch_conv3<16>(pl.a_hi, pl.a_lo, o_hi, o_lo, p, smem, st);
    case 32: return launch_conv3<32>(pl.a_hi, pl.a_lo, o_hi, o_lo, p, smem, st);
    case 48: return launch_conv3<48>(pl.a_hi, pl.a_lo, o_hi, o_lo, p, smem, st);
    case 64: return launch_conv3<64>(pl.a_hi, pl.a_lo, o_hi, o_lo, p, smem, st);
    case 80: return launch_conv3<80>(pl.a_hi, pl.a_lo, o_hi, o_lo, p, smem, st);
  }
  set_error("umma_conv: n_c=%d has no kernel instance", n_c);
  return B200SEP_ERR_ARG;
}

static int pick_nc(int Cout, int mult, int limit) {  // largest n_c | Cout with mult*n_c <= limit and mult*n_c % 16 == 0
  for (int nc = Cout; nc >= 4; --nc)
    if (Cout % nc == 0 && mult * nc <= limit && (mult * nc) % 16 == 0 && nc % 16 == 0) return nc;
  return 0;
}
bool umma_updown_supported(int Cin, int Cout, int F_in, int up) {
  return Cin % 16 == 0 && F_in % 8 == 0 && pick_nc(Cout, up ? 4 : 2, 256) > 0 && (up || F_in % 2 == 0);
}
int umma_updown_choose(int Cin, int Cout, int up, int* kc, int* n_c) {
  int k = 64;
  while (k > 16 && Cin % k != 0) k -= 16;
  if (Cin % 48 == 0) k = 48;
  *kc = k;
  *n_c = pick_nc(Cout, up ? 4 : 2, up ? 192 : 256);
  if (*n_c == 0) *n_c = pick_nc(Cout, up ? 4 : 2, 256);
  return 0;
}

// x: pair (B, Cin, T, F) -> ConvTranspose2d(k2,s2)+BN+ReLU (* skip) -> pair (B, Cout, 2T, 2F)
int umma_up_run(const UmmaConvPlan& pl, const void* wb_hi, const void* wb_lo, int B, int Cout, int n_c, const float* scale, const float* shift, int relu,
                const void* skip_hi, const void* skip_lo, void* out_hi, void* out_lo, cudaStream_t st) {
  UmmaEpilogue e;
  e.scale = scale; e.shift = shift; e.act = relu ? 1 : 0; e.out_hi = out_hi; e.out_lo = out_lo; e.res_hi = skip_hi; e.res_lo = skip_lo;
  return umma_up_run_ex(pl, wb_hi, wb_lo, B, Cout, n_c, e, st);
}

int umma_up_run_ex(const UmmaConvPlan& pl, const void* wb_hi, const void* wb_lo, int B, int Cout, int n_c, const UmmaEpilogue& e, cudaStream_t st) {
  UmmaParams p{};
  p.mode = 2; p.f_stride = kTileM; p.t_mul = 1; p.t_off = 0;
  p.n_c = n_c; p.n_tile = 4 * n_c; p.n_total = Cout;
  p.kc = pl.kc; p.n_chunks = pl.Cin / pl.kc; p.num_iters = p.n_chunks; p.ksteps = pl.kc / 16;
  p.a_bytes = (uint32_t)pl.kc * 256; p.b_bytes = (uint32_t)p.ksteps * p.n_tile * 32;
  p.T = pl.T; p.F = pl.F; p.Cin = pl.Cin; p.Cout = Cout; p.n_tiles = Cout / n_c;
  p.wb_hi = (const bf16*)wb_hi; p.wb_lo = (const bf16*)wb_lo;
  fill_epilogue(p, e, Cout);
  dim3 grid(cdiv(pl.F, kTileM), pl.T, B * p.n_tiles);
  return launch(pl.a_hi, pl.a_lo, pl.a_hi, pl.a_lo, p, grid, st);
}

// x: pair (B, Cin, T, F) -> Conv2d(k2,s2)+BN+ReLU -> pair (B, Cout, T/2, F/2)
int umma_down_run(const UmmaConvPlan& pl, const void* wb_hi, const void* wb_lo, int B, int Cout, int n_c, const float* scale, const float* shift, int relu,
                  void* out_hi, void* out_lo, cudaStream_t st) {
  UmmaEpilogue e;
  e.scale = scale; e.shift = shift; e.act = relu ? 1 : 0; e.out_hi = out_hi; e.out_lo = out_lo;
  return umma_down_run_ex(pl, wb_hi, wb_lo, B, Cout, n_c, e, st);
}

int umma_down_run_ex(const UmmaConvPlan& pl, const void* wb_hi, const void* wb_lo, int B, int Cout, int n_c, const UmmaEpilogue& e, cudaStream_t st) {
  UmmaParams p{};
  p.mode = 3; p.f_stride = kTileM; p.t_mul = 2; p.t_off = 0;
  p.n_c = n_c; p.n_tile = 2 * n_c; p.n_total = Cout;
  p.kc = pl.kc; p.n_chunks = pl.Cin / pl.kc; p.num_iters = 2 * p.n_chunks; p.ksteps = pl.kc / 16;
  p.a_bytes = (uint32_t)pl.kc * 256; p.b_bytes = (uint32_t)p.ksteps * p.n_tile * 32;
  p.T = pl.T; p.F = pl.F; p.Cin = pl.Cin; p.Cout = Cout; p.n_tiles = Cout / n_c;
  p.wb_hi = (const bf16*)wb_hi; p.wb_lo = (const bf16*)wb_lo;
  fill_epilogue(p, e, Cout);
  dim3 grid(cdiv(pl.F, kTileM), pl.T / 2, B * p.n_tiles);
  return launch(pl.a_hi, pl.a_lo, pl.a_hi, pl.a_lo, p, grid, st);
}

// Generic blocking: value(row, r, ci) for B rows [rows], row taps [n_r], -> [Cout/n_c][r][Cin/kc][kc/16][rows x 16 core-matrix tiled]
template <class F>
static void block_weights(int n_tiles, int n_r, int Cin, int kc, int rows, F value, std::vector<uint16_t>& hi, std::vector<uint16_t>& lo) {
  auto f2bf = [](float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
  };
  auto bf2f = [](uint16_t h) {
    uint32_t u = (uint32_t)h << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
  };
  const int n_chunks = Cin / kc, ksteps = kc / 16;
  hi.assign((size_t)n_tiles * n_r * Cin * rows, 0);
  lo.assign(hi.size(), 0);
  size_t pos = 0;
  for (int nt = 0; nt < n_tiles; ++nt)
    for (int r = 0; r < n_r; ++r)
      for (int ch = 0; ch < n_chunks; ++ch)
        for (int j = 0; j < ksteps; ++j) {
          for (int row = 0; row < rows; ++row)
            for (int kk = 0; kk < 16; ++kk) {
              const float v = value(nt, row, r, ch * kc + j * 16 + kk);
              const size_t o = pos + (size_t)((row / 8) * 2 + kk / 8) * 64 + (row % 8) * 8 + (kk % 8);
              hi[o] = f2bf(v);
              lo[o] = f2bf(v - bf2f(hi[o]));
            }
          pos += (size_t)rows * 16;
        }
}
// ConvTranspose2d weight (Cin, Cout, 2, 2): B rows = (q = dy*2+dx, co_local)
void umma_up_block_weights(const float* w, int Cin, int Cout, int kc, int n_c, std::vector<uint16_t>& hi, std::vector<uint16_t>& lo) {
  block_weights(Cout / n_c, 1, Cin, kc, 4 * n_c, [&](int nt, int row, int, int ci) {
    const int q = row / n_c, co = nt * n_c + row % n_c;
    return w[((size_t)ci * Cout + co) * 4 + q];
  }, hi, lo);
}
// Conv2d weight (Cout, Cin, 2, 2) stride 2: row taps r = dy, B rows = (dx, co_local)
void umma_down_block_weights(const float* w, int Cout, int Cin, int kc, int n_c, std::vector<uint16_t>& hi, std::vector<uint16_t>& lo) {
  block_weights(Cout / n_c, 2, Cin, kc, 2 * n_c, [&](int nt, int row, int dy, int ci) {
    const int dx = row / n_c, co = nt * n_c + row % n_c;
    return w[(((size_t)co * Cin + ci) * 2 + dy) * 2 + dx];
  }, hi, lo);
}

// Conv2d weight (Cout, Cin, 1, 1): one tap, B rows = co_local
void umma_pw_block_weights(const float* w, int Cout, int Cin, int kc, int n_c, std::vector<uint16_t>& hi, std::vector<uint16_t>& lo) {
  block_weights(Cout / n_c, 1, Cin, kc, n_c, [&](int nt, int row, int, int ci) { return w[(size_t)(nt * n_c + row) * Cin + ci]; }, hi, lo);
}
bool umma_pw_supported(int Cin, int Cout, int F) { return Cin % 16 == 0 && Cout % 16 == 0 && F % 8 == 0; }
int umma_pw_choose(int Cin, int Cout, int* kc, int* n_c) {
  int k = 64;
  while (k > 16 && Cin % k != 0) k -= 16;
  if (Cin % 48 == 0) k = 48;
  *kc = k;
  *n_c = pick_nc(Cout, 1, 256);
  return 0;
}
// x: pair (B, Cin, T, F) -> Conv2d 1x1 (+affine, act, +res, *mul) -> pair or fp32 (B, Cout, T, F)
int umma_pw_run_ex(const UmmaConvPlan& pl, const void* wb_hi, const void* wb_lo, int B, int Cout, int n_c, const UmmaEpilogue& e, cudaStream_t st) {
  UmmaParams p{};
  p.mode = 4; p.f_stride = kTileM; p.t_mul = 1; p.t_off = 0;
  p.n_c = n_c; p.n_tile = n_c; p.n_total = Cout;
  p.kc = pl.kc; p.n_chunks = pl.Cin / pl.kc; p.num_iters = p.n_chunks; p.ksteps = pl.kc / 16;
  p.a_bytes = (uint32_t)pl.kc * 256; p.b_bytes = (uint32_t)p.ksteps * p.n_tile * 32;
  p.T = pl.T; p.F = pl.F; p.Cin = pl.Cin; p.Cout = Cout; p.n_tiles = Cout / n_c;
  p.wb_hi = (const bf16*)wb_hi; p.wb_lo = (const bf16*)wb_lo;
  fill_epilogue(p, e, Cout);
  dim3 grid(cdiv(pl.F, kTileM), pl.T, B * p.n_tiles);
  return launch(pl.a_hi, pl.a_lo, pl.a_hi, pl.a_lo, p, grid, st);
}

// Host-side blocking of a (Cout, Cin, 3, 3) fp32 filter into the B operand stream of umma_conv_run:
// [Cout/n_c][dy][Cin/kc][kc/16] blocks of [3*n_c rows = (dx, co)][16 k] stored as 8x8 core matrices (K-major, no swizzle).
void umma_conv_block_weights(const float* w, int Cout, int Cin, int kc, int n_c, std::vector<uint16_t>& hi, std::vector<uint16_t>& lo) {
  auto f2bf = [](float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    u += 0x7fffu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
  };
  auto bf2f = [](uint16_t h) {
    uint32_t u = (uint32_t)h << 16;
    float f;
    memcpy(&f, &u, 4);
    return f;
  };
  const int n_tiles = Cout / n_c, n_chunks = Cin / kc, ksteps = kc / 16, rows = 3 * n_c;
  hi.assign((size_t)Cout * Cin * 9, 0);
  lo.assign(hi.size(), 0);
  size_t pos = 0;
  for (int nt = 0; nt < n_tiles; ++nt)
    for (int dy = 0; dy < 3; ++dy)
      for (int ch = 0; ch < n_chunks; ++ch)
        for (int j = 0; j < ksteps; ++j) {
          for (int r = 0; r < rows; ++r)
            for (int kk = 0; kk < 16; ++kk) {
              const int dx = r / n_c, co = nt * n_c + r % n_c, ci = ch * kc + j * 16 + kk;
              const float v = w[(((size_t)co * Cin + ci) * 3 + dy) * 3 + dx];
              const size_t o = pos + (size_t)((r / 8) * 2 + kk / 8) * 64 + (r % 8) * 8 + (kk % 8);
              hi[o] = f2bf(v);
              lo[o] = f2bf(v - bf2f(hi[o]));
            }
          pos += (size_t)rows * 16;
        }
}

// ---------------------------------------------------------------------------------------------------------
// pair <-> fp32 helpers
__global__ void split_pair_kernel(const float* __restrict__ x, bf16* __restrict__ hi, bf16* __restrict__ lo, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) split_store2(x[i], hi[i], lo[i]);
}
__global__ void join_pair_kernel(const bf16* __restrict__ hi, const bf16* __restrict__ lo, float* __restrict__ y, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    y[i] = __bfloat162float(hi[i]) + __bfloat162float(lo[i]);
}
int split_pair(const float* x, void* hi, void* lo, int64_t n, cudaStream_t st) {
  if (n == 0) return B200SEP_OK;
  split_pair_kernel<<<(int)std::min<int64_t>(cdiv(n, 1024), kNumSMs * 8), 256, 0, st>>>(x, (bf16*)hi, (bf16*)lo, n);
  B2_LAUNCHED();
  return B200SEP_OK;
}
int join_pair(const void* hi, const void* lo, float* y, int64_t n, cudaStream_t st) {
  if (n == 0) return B200SEP_OK;
  join_pair_kernel<<<(int)std::min<int64_t>(cdiv(n, 1024), kNumSMs * 8), 256, 0, st>>>((const bf16*)hi, (const bf16*)lo, y, n);
  B2_LAUNCHED();
  return B200SEP_OK;
}

}  // namespace b200sep

// ---------------------------------------------------------------------------------------------------------
// self-test entry points (exported through the C ABI so the GPU test-suite can check each tensor-core operator in
// isolation against a plain fp32 reference): fp32 in -> split -> tcgen05 op -> join -> fp32 out.
using namespace b200sep;

extern "C" int b200sep_selftest_umma_gemm(const float* a, const float* w, const float* res, float* out, int M, int N, int K, int rows_per_channel,
                                          int channels, const float* scale, const float* shift, int relu, void* stream) {
  B2_CHECK_ARG(a && w && out && scale && shift, "selftest_umma_gemm: NULL argument");
  B2_CHECK_ARG(umma_gemm_supported(M, N, K), "selftest_umma_gemm: shape M=%d N=%d K=%d not supported by the tensor-core path", M, N, K);
  cudaStream_t st = (cudaStream_t)stream;
  uint16_t *a_p = nullptr, *w_p = nullptr, *o_p = nullptr, *r_p = nullptr;
  const int64_t na = (int64_t)M * K, nw = (int64_t)N * K, no = (int64_t)M * N;
  B2_CUDA(cudaMalloc(&a_p, na * 4));
  B2_CUDA(cudaMalloc(&w_p, nw * 4));
  B2_CUDA(cudaMalloc(&o_p, no * 4));
  if (res) B2_CUDA(cudaMalloc(&r_p, no * 4));
  int rc = split_pair(a, a_p, a_p + na, na, st);
  if (!rc) rc = split_pair(w, w_p, w_p + nw, nw, st);
  if (!rc && res) rc = split_pair(res, r_p, r_p + no, no, st);
  UmmaGemmPlan pl;
  if (!rc) rc = umma_gemm_plan_create(&pl, a_p, a_p + na, w_p, w_p + nw, M, N, K);
  if (!rc) rc = umma_gemm_run(pl, scale, shift, rows_per_channel, channels, relu, o_p, o_p + no, r_p, r_p ? r_p + no : nullptr, M, st);
  if (!rc) rc = join_pair(o_p, o_p + no, out, no, st);
  cudaStreamSynchronize(st);
  cudaFree(a_p); cudaFree(w_p); cudaFree(o_p);
  if (r_p) cudaFree(r_p);
  return rc;
}

extern "C" int b200sep_selftest_umma_conv3x3(const float* x, const float* w_host, float* out, int B, int Cin, int Cout, int T, int F, const float* scale,
                                             const float* shift, int relu, void* stream) {
  B2_CHECK_ARG(x && w_host && out && scale && shift, "selftest_umma_conv3x3: NULL argument");
  B2_CHECK_ARG(umma_conv_supported(Cin, Cout, F, 3, 3), "selftest_umma_conv3x3: Cin=%d Cout=%d F=%d not supported by the tensor-core path", Cin, Cout, F);
  cudaStream_t st = (cudaStream_t)stream;
  int kc, n_c;
  umma_conv_choose(Cin, Cout, &kc, &n_c);
  std::vector<uint16_t> hi, lo;
  umma_conv_block_weights(w_host, Cout, Cin, kc, n_c, hi, lo);
  uint16_t *x_p = nullptr, *o_p = nullptr, *w_p = nullptr;
  const int64_t nx = (int64_t)B * Cin * T * F, no = (int64_t)B * Cout * T * F, nw = (int64_t)hi.size();
  B2_CUDA(cudaMalloc(&x_p, nx * 4));
  B2_CUDA(cudaMalloc(&o_p, no * 4));
  B2_CUDA(cudaMalloc(&w_p, nw * 4));
  B2_CUDA(cudaMemcpy(w_p, hi.data(), nw * 2, cudaMemcpyHostToDevice));
  B2_CUDA(cudaMemcpy(w_p + nw, lo.data(), nw * 2, cudaMemcpyHostToDevice));
  int rc = split_pair(x, x_p, x_p + nx, nx, st);
  UmmaConvPlan pl;
  if (!rc) rc = umma_conv_plan_create(&pl, x_p, x_p + nx, B, Cin, T, F, kc);
  if (!rc) rc = umma_conv_run(pl, w_p, w_p + nw, B, Cout, n_c, 3, scale, shift, relu, o_p, o_p + no, st);
  if (!rc) rc = join_pair(o_p, o_p + no, out, no, st);
  cudaStreamSynchronize(st);
  cudaFree(x_p); cudaFree(o_p); cudaFree(w_p);
  return rc;
}

extern "C" int b200sep_selftest_umma_updown(const float* x, const float* w_host, const float* skip, float* out, int B, int Cin, int Cout, int T, int F,
                                            const float* scale, const float* shift, int relu, int up, void* stream) {
  B2_CHECK_ARG(x && w_host && out && scale && shift, "selftest_umma_updown: NULL argument");
  B2_CHECK_ARG(umma_updown_supported(Cin, Cout, F, up), "selftest_umma_updown: Cin=%d Cout=%d F=%d not supported by the tensor-core path", Cin, Cout, F);
  cudaStream_t st = (cudaStream_t)stream;
  int kc, n_c;
  umma_updown_choose(Cin, Cout, up, &kc, &n_c);
  std::vector<uint16_t> hi, lo;
  if (up) umma_up_block_weights(w_host, Cin, Cout, kc, n_c, hi, lo);
  else umma_down_block_weights(w_host, Cout, Cin, kc, n_c, hi, lo);
  uint16_t *x_p = nullptr, *o_p = nullptr, *w_p = nullptr, *s_p = nullptr;
  const int64_t nx = (int64_t)B * Cin * T * F, no = up ? (int64_t)B * Cout * 4 * T * F : (int64_t)B * Cout * (T / 2) * (F / 2), nw = (int64_t)hi.size();
  B2_CUDA(cudaMalloc(&x_p, nx * 4));
  B2_CUDA(cudaMalloc(&o_p, no * 4));
  B2_CUDA(cudaMalloc(&w_p, nw * 4));
  if (skip) B2_CUDA(cudaMalloc(&s_p, no * 4));
  B2_CUDA(cudaMemcpy(w_p, hi.data(), nw * 2, cudaMemcpyHostToDevice));
  B2_CUDA(cudaMemcpy(w_p + nw, lo.data(), nw * 2, cudaMemcpyHostToDevice));
  int rc = split_pair(x, x_p, x_p + nx, nx, st);
  if (!rc && skip) rc = split_pair(skip, s_p, s_p + no, no, st);
  UmmaConvPlan pl;
  if (!rc) rc = umma_conv_plan_create(&pl, x_p, x_p + nx, B, Cin, T, F, kc);
  if (!rc) {
    if (up) rc = umma_up_run(pl, w_p, w_p + nw, B, Cout, n_c, scale, shift, relu, s_p, s_p ? s_p + no : nullptr, o_p, o_p + no, st);
    else rc = umma_down_run(pl, w_p, w_p + nw, B, Cout, n_c, scale, shift, relu, o_p, o_p + no, st);
  }
  if (!rc) rc = join_pair(o_p, o_p + no, out, no, st);
  cudaStreamSynchronize(st);
  cudaFree(x_p); cudaFree(o_p); cudaFree(w_p);
  if (s_p) cudaFree(s_p);
  return rc;
}

// Every epilogue option of the conv modes as MDX23C uses them (tfc_net.cu): act, residual (multiplied for UP), multiplier, output channel slice, fp32 store.
// `out` is split into the pair buffer before the run and joined back after it, so the channels outside the slice must come back unchanged.
extern "C" int b200sep_selftest_umma_ex(int kind, const float* x, const float* w_host, const float* res, const float* mul, float* out, int B, int Cin, int Cout,
                                        int T, int F, int act, int out_c_total, int out_c_off, int out_f32, void* stream) {
  B2_CHECK_ARG(x && w_host && out, "selftest_umma_ex: NULL argument");
  B2_CHECK_ARG(kind >= 0 && kind <= 3 && act >= 0 && act <= 2 && B >= 1 && T >= 1, "selftest_umma_ex: bad kind=%d / act=%d / B=%d / T=%d", kind, act, B, T);
  const int ct = out_c_total > 0 ? out_c_total : Cout;
  B2_CHECK_ARG(out_c_off >= 0 && out_c_off + Cout <= ct, "selftest_umma_ex: channels [%d, %d) do not fit in %d", out_c_off, out_c_off + Cout, ct);
  B2_CHECK_ARG(!mul || kind <= 1, "selftest_umma_ex: the multiplier exists for conv3x3 and pw only");
  B2_CHECK_ARG(!res || kind != 2, "selftest_umma_ex: the down conv has no residual");
  B2_CHECK_ARG(!out_f32 || kind == 1, "selftest_umma_ex: the fp32 store exists for pw only");
  int kc = 0, n_c = 0, To = T, Fo = F;
  std::vector<uint16_t> hi, lo;
  if (kind == 0) {
    B2_CHECK_ARG(umma_conv_supported(Cin, Cout, F, 3, 3), "selftest_umma_ex: conv3x3 Cin=%d Cout=%d F=%d not supported by the tensor-core path", Cin, Cout, F);
    umma_conv_choose(Cin, Cout, &kc, &n_c);
    umma_conv_block_weights(w_host, Cout, Cin, kc, n_c, hi, lo);
  } else if (kind == 1) {
    B2_CHECK_ARG(umma_pw_supported(Cin, Cout, F), "selftest_umma_ex: pw Cin=%d Cout=%d F=%d not supported by the tensor-core path", Cin, Cout, F);
    umma_pw_choose(Cin, Cout, &kc, &n_c);
    umma_pw_block_weights(w_host, Cout, Cin, kc, n_c, hi, lo);
  } else {
    const int up = kind == 3;
    B2_CHECK_ARG(umma_updown_supported(Cin, Cout, F, up) && (up || T % 2 == 0), "selftest_umma_ex: %s Cin=%d Cout=%d T=%d F=%d not supported by the tensor-core path",
                 up ? "up" : "down", Cin, Cout, T, F);
    umma_updown_choose(Cin, Cout, up, &kc, &n_c);
    if (up) umma_up_block_weights(w_host, Cin, Cout, kc, n_c, hi, lo);
    else umma_down_block_weights(w_host, Cout, Cin, kc, n_c, hi, lo);
    To = up ? 2 * T : T / 2;
    Fo = up ? 2 * F : F / 2;
  }
  cudaStream_t st = (cudaStream_t)stream;
  uint16_t *x_p = nullptr, *o_p = nullptr, *w_p = nullptr, *r_p = nullptr, *m_p = nullptr;
  const int64_t nx = (int64_t)B * Cin * T * F, no = (int64_t)B * ct * To * Fo, nr = (int64_t)B * Cout * To * Fo, nw = (int64_t)hi.size();
  B2_CUDA(cudaMalloc(&x_p, nx * 4));
  B2_CUDA(cudaMalloc(&w_p, nw * 4));
  if (!out_f32) B2_CUDA(cudaMalloc(&o_p, no * 4));
  if (res) B2_CUDA(cudaMalloc(&r_p, nr * 4));
  if (mul) B2_CUDA(cudaMalloc(&m_p, nr * 4));
  B2_CUDA(cudaMemcpy(w_p, hi.data(), nw * 2, cudaMemcpyHostToDevice));
  B2_CUDA(cudaMemcpy(w_p + nw, lo.data(), nw * 2, cudaMemcpyHostToDevice));
  int rc = split_pair(x, x_p, x_p + nx, nx, st);
  if (!rc && o_p) rc = split_pair(out, o_p, o_p + no, no, st);
  if (!rc && r_p) rc = split_pair(res, r_p, r_p + nr, nr, st);
  if (!rc && m_p) rc = split_pair(mul, m_p, m_p + nr, nr, st);
  UmmaConvPlan pl;
  if (!rc) rc = umma_conv_plan_create(&pl, x_p, x_p + nx, B, Cin, T, F, kc);
  UmmaEpilogue e;
  e.act = act;
  if (o_p) { e.out_hi = o_p; e.out_lo = o_p + no; }
  else e.out_f32 = out;
  if (r_p) { e.res_hi = r_p; e.res_lo = r_p + nr; }
  if (m_p) { e.mul_hi = m_p; e.mul_lo = m_p + nr; }
  e.out_c_total = ct;
  e.out_c_off = out_c_off;
  if (!rc) {
    if (kind == 0) rc = umma_conv_run_ex(pl, w_p, w_p + nw, B, Cout, n_c, e, st);
    else if (kind == 1) rc = umma_pw_run_ex(pl, w_p, w_p + nw, B, Cout, n_c, e, st);
    else if (kind == 2) rc = umma_down_run_ex(pl, w_p, w_p + nw, B, Cout, n_c, e, st);
    else rc = umma_up_run_ex(pl, w_p, w_p + nw, B, Cout, n_c, e, st);
  }
  if (!rc && o_p) rc = join_pair(o_p, o_p + no, out, no, st);
  cudaStreamSynchronize(st);
  cudaFree(x_p); cudaFree(w_p);
  if (o_p) cudaFree(o_p);
  if (r_p) cudaFree(r_p);
  if (m_p) cudaFree(m_p);
  return rc;
}
