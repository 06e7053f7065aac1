/*
 * b200sep.h -- C ABI of the B200-native stem-separation hot path (libb200sep.so, sm_100a only).
 *
 * The reference (nomadkaraoke/python-audio-separator v0.44.1) is pure Python; its hot path calls into
 * third-party wheels (ATen FFT/conv, onnxruntime).  This header is the FFI a maintainer would bind in place
 * of those calls (ctypes stub: INTEGRATION.md).  Each entry point cites the reference interface it replaces
 * (paths relative to the reference root).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; sizes are element counts;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are asynchronous;
 *   - return value: 0 = ok, negative = error (b200sep_last_error() gives the text, thread-local);
 *   - no exceptions, no torch types, no ownership transfer except b200sep_*_create / _destroy handles;
 *   - there is no CPU fallback: without a CUDA device every compute entry point returns B200SEP_ERR_CUDA.
 */
#ifndef B200SEP_H
#define B200SEP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200SEP_OK 0
#define B200SEP_ERR_ARG (-1)     /* bad argument / unsupported shape */
#define B200SEP_ERR_CUDA (-2)    /* CUDA runtime error (launch, alloc, no device) */
#define B200SEP_ERR_STATE (-3)   /* handle used before it was fully initialised */

#define B200SEP_ABI_VERSION 1

/* spectrogram memory layouts */
#define B200SEP_LAYOUT_CFT 0 /* (B, 2C, dim_f, frames): the reference's STFT.__call__ layout (uvr_lib_v5/stft.py:44-56) */
#define B200SEP_LAYOUT_CTF 1 /* (B, 2C, frames, dim_f): what ConvTDFNet computes on after transpose(-1,-2) (uvr_lib_v5/mdxnet.py:101) */

int b200sep_abi_version(void);
const char* b200sep_last_error(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches evidence) */
uint64_t b200sep_launch_count(void);

/* ---------------------------------------------------------------------------------------------------
 * STFT plan: twiddle / window tables for one (n_fft, hop) pair.  n_fft must factor into {2,3,5}.
 * Replaces STFT.__init__ (uvr_lib_v5/stft.py:11-18).
 */
typedef struct b200sep_stft_plan b200sep_stft_plan;
int b200sep_stft_plan_create(b200sep_stft_plan** plan, int n_fft, int hop);
void b200sep_stft_plan_destroy(b200sep_stft_plan* plan);

/*
 * Forward STFT of `batch` stereo chunks.  Replaces STFT.__call__ (uvr_lib_v5/stft.py:20-56): periodic Hann,
 * center=True with reflect padding of n_fft/2, one-sided, un-normalised, planes [L_re, L_im, R_re, R_im],
 * frequency axis cropped to dim_f; bins [0, zero_bins) are written as 0 (fuses `spek[:, :, :3, :] *= 0`,
 * architectures/mdx_separator.py:425).
 *
 * Chunk b, channel c, sample n is read from  wave[b*batch_stride + c*chan_stride + n]  when valid_len <= 0 or
 * b*batch_stride + n < valid_len, and is 0 otherwise (fuses the right zero-padding of the short last chunk,
 * mdx_separator.py:363-366).  Two addressings are used:
 *   - a contiguous (B,2,T) tensor:            batch_stride = 2T,   chan_stride = T, valid_len = 0 (unlimited);
 *   - chunks cut out of a padded (2,L) mixture: batch_stride = step, chan_stride = L, valid_len = L - offset of `wave`.
 * `chunk_len` = T must be > n_fft/2 (reflect padding); frames = T/hop + 1 (integer division, like torch.stft).
 * spec: layout CFT or CTF, float32, batch*4*dim_f*frames elements.
 */
int b200sep_stft_forward(const b200sep_stft_plan* plan, const float* wave, int64_t batch_stride, int64_t chan_stride,
                         int64_t valid_len, int batch, int chunk_len, int dim_f, int zero_bins, int layout,
                         float* spec, void* stream);

/*
 * Inverse STFT.  Replaces STFT.inverse (uvr_lib_v5/stft.py:99-126): bins dim_f..n_fft/2 zero-filled, complex
 * irfft per frame, Hann window, overlap-add at hop, division by the overlap-added squared window, n_fft/2
 * trimmed from both ends.  spec (B,4,dim_f,frames) [CFT] or (B,4,frames,dim_f) [CTF] -> wave (B,2,hop*(frames-1)).
 * `work` must hold b200sep_stft_inverse_work_floats(...) floats.
 */
int64_t b200sep_stft_inverse_work_floats(const b200sep_stft_plan* plan, int batch, int frames, int dim_f, int layout);
int b200sep_stft_inverse(const b200sep_stft_plan* plan, const float* spec, int batch, int frames, int dim_f, int layout,
                         float* wave, float* work, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Windowed overlap-add of the per-chunk outputs.  Replaces the accumulation loop + divide + trim of
 * MDXSeparator.demix (architectures/mdx_separator.py:339-340, :348-401):
 *
 *   result[:, s_i : e_i] += y_i[:, :e_i-s_i] * hanning(e_i - s_i);  divider[...] += hanning(e_i - s_i)
 *   out = (result / divider)[:, trim : trim + n_out] * out_scale
 *
 * with s_i = i*step, e_i = min(s_i + chunk_len, total_len), written as a deterministic gather (each output
 * sample sums its <= ceil(chunk/step) covering chunks in chunk order).  use_window=0 reproduces overlap==0
 * (divider += 1).  chunks: (n_chunks, 2, chunk_len) float32; out: (2, n_out) float32.
 * If mix != NULL (2, n_out), also writes secondary = mix - compensate * out  (mdx_separator.py:182),
 * both as (n_out, 2) interleaved when interleave != 0 (the `.T` of mdx_separator.py:163) else (2, n_out).
 */
int b200sep_demix_overlap_add(const float* chunks, int n_chunks, int chunk_len, int64_t step, int64_t total_len,
                              int64_t trim, int64_t n_out, int use_window, float out_scale, const float* mix,
                              float compensate, int interleave, float* primary, float* secondary, void* stream);

/*
 * Same, for ONE rank of a time-sharded run (chunk ranges split across GPUs): `chunks` holds the n_local_chunks chunks
 * [first_chunk, first_chunk + n_local_chunks) of the global n_chunks grid (own chunks plus the halo received from the
 * left neighbour) and only outputs q in [q_begin, q_end) are written; primary / secondary / mix are still indexed
 * with the global q and n_out.  Returns B200SEP_ERR_ARG if a covering chunk is missing from the buffer.
 */
int b200sep_demix_overlap_add_range(const float* chunks, int first_chunk, int n_local_chunks, int n_chunks, int chunk_len, int64_t step,
                                    int64_t total_len, int64_t trim, int64_t n_out, int64_t q_begin, int64_t q_end, int use_window,
                                    float out_scale, const float* mix, float compensate, int interleave, float* primary,
                                    float* secondary, void* stream);
/* Same with the outputs and the mix given as SLICES: primary / secondary hold the rows [out_base, ...) of the interleaved (n_out, 2) stems and
 * mix is (2, mix_ld) holding the samples [mix_base, mix_base + mix_ld) -- a rank of the sharded end-to-end path only ever holds its own part. */
int b200sep_demix_overlap_add_range_ex(const float* chunks, int first_chunk, int n_local_chunks, int n_chunks, int chunk_len, int64_t step,
                                       int64_t total_len, int64_t trim, int64_t n_out, int64_t q_begin, int64_t q_end, int use_window,
                                       float out_scale, const float* mix, int64_t mix_ld, int64_t mix_base, float compensate, int interleave,
                                       float* primary, float* secondary, int64_t out_base, void* stream);

/* max |x| over n floats -> *result (device float).  (np.abs(mix).max(), mdx_separator.py:155; spec_utils.py:110) */
int b200sep_absmax(const float* x, int64_t n, float* result, void* stream);
/* y = x * s where s = max_peak/absmax if absmax > max_peak; min_peak/absmax if min_peak>=0 and absmax < min_peak;
 * else 1 (spec_utils.normalize, uvr_lib_v5/spec_utils.py:99-115).  absmax is a device scalar. */
int b200sep_normalize(const float* x, int64_t n, const float* absmax, float max_peak, float min_peak, float* y, void* stream);
/* (x*32767) truncated toward zero to int16 (common_separator.py:331); x is (n,) float32 */
int b200sep_to_pcm16(const float* x, int64_t n, int16_t* y, void* stream);
/* The same at the input file's bit depth (common_separator.py:322-383): n samples -> n * bits/8 little-endian bytes.  via_int16 = 1: the default (pydub) writer,
 * int16 quantisation widened by shifting; 0: the libsndfile writer, lrint(x * (2^(bits-1) - 1)). */
int b200sep_to_pcm_bytes(const float* x, int64_t n, int bits, int via_int16, uint8_t* y, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * ConvTDFNet (the graph inside UVR-MDX-NET-*.onnx; topology: uvr_lib_v5/mdxnet.py:30-120, modules.py:1-74).
 * Replaces `self.model_run(spek)` = ort.InferenceSession.run (architectures/mdx_separator.py:122-123, :443).
 *
 * The host passes the raw parameters in the reference module's state_dict order (see
 * b200sep_mdxnet_param_count / the Python loader); BatchNorm folding, weight re-layout and the bf16 hi/lo
 * split for the tensor-core path happen once at create time on the device.
 */
typedef struct b200sep_mdxnet b200sep_mdxnet;
typedef struct {
  int32_t dim_c;      /* 4 */
  int32_t dim_f;      /* 3072 */
  int32_t dim_t;      /* 256 */
  int32_t num_blocks; /* 11 */
  int32_t l;          /* 3 convs per TFC */
  int32_t g;          /* 48 growth */
  int32_t k;          /* 3 */
  int32_t bn;         /* 8 TDF bottleneck factor */
  int32_t max_batch;  /* chunks per forward the workspace is sized for */
  int32_t precision;  /* 0 = fp32 SIMT everywhere; 1 = bf16x3 split tcgen05 where profitable */
} b200sep_mdxnet_config;

/* number of float parameters expected in `params_host` for this config */
int64_t b200sep_mdxnet_param_count(const b200sep_mdxnet_config* cfg);
int b200sep_mdxnet_create(b200sep_mdxnet** net, const b200sep_mdxnet_config* cfg, const float* params_host, int64_t n_params);
void b200sep_mdxnet_destroy(b200sep_mdxnet* net);
/* bytes of device memory held by the handle (weights + activation workspace) */
int64_t b200sep_mdxnet_device_bytes(const b200sep_mdxnet* net);
/*
 * Forward: spec_in (B,4,dim_t,dim_f) [CTF] or (B,4,dim_f,dim_t) [CFT] float32 -> spec_out, same shape/layout.
 * batch <= max_batch.
 */
int b200sep_mdxnet_forward(b200sep_mdxnet* net, const float* spec_in, float* spec_out, int batch, int layout, void* stream);

/*
 * Optional device-side timing of the forward, by kernel category (measurement only; bench.py's roofline).
 * enable!=0 clears the records and makes every subsequent forward record a CUDA-event pair around each launch on
 * the caller's stream; _read synchronises on those events and returns, per category, the summed device time,
 * launch count and the ALGORITHMIC flops (2*MAC, unpadded) and bytes (inputs + outputs + weights, fp32) of the
 * launches recorded.  Returns the number of categories (names via _profile_name).
 */
int b200sep_mdxnet_profile_enable(b200sep_mdxnet* net, int enable);
int b200sep_mdxnet_profile_read(b200sep_mdxnet* net, int max_categories, float* ms, int64_t* launches, double* flops, double* bytes);
const char* b200sep_mdxnet_profile_name(int category);

/* ---------------------------------------------------------------------------------------------------
 * Whole-chunk operator: STFT -> zero bins -> net (optionally denoise: 0.5*f(x) - 0.5*f(-x)) -> iSTFT.
 * Replaces MDXSeparator.run_model (architectures/mdx_separator.py:414-450) for `batch` chunks whose samples
 * are read straight out of the padded mixture (see b200sep_stft_forward addressing).
 * net == NULL reproduces is_match_mix=True (mdx_separator.py:429-432).  wave_out: (batch, 2, chunk_len).
 */
int64_t b200sep_mdx_run_model_work_floats(const b200sep_stft_plan* plan, int batch, int chunk_len, int dim_f);
int b200sep_mdx_run_model(const b200sep_stft_plan* plan, b200sep_mdxnet* net, const float* wave, int64_t batch_stride,
                          int64_t chan_stride, int64_t valid_len, int batch, int chunk_len, int dim_f, int denoise,
                          float* wave_out, float* work, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * TFC_TDF_net (MDX23C; uvr_lib_v5/tfc_tdf_v3.py:151-267).  Replaces `self.model_run(batch)` of the non-Roformer MDXC branch
 * (architectures/mdxc_separator.py:390) between its two STFTs.  Only norm = InstanceNorm (affine), act = gelu, scale = [2, 2]
 * (the MDX23C-8KFFT-InstVoc_HQ configuration).  Parameters in the reference module's state_dict order.
 */
typedef struct b200sep_tfcnet b200sep_tfcnet;
typedef struct {
  int32_t dim_f;          /* audio.dim_f (4096) */
  int32_t dim_t;          /* frames per chunk (inference.dim_t, 256) */
  int32_t num_subbands;   /* model.num_subbands (4) */
  int32_t audio_channels; /* audio.num_channels (2) */
  int32_t num_scales;     /* 5 */
  int32_t l;              /* num_blocks_per_scale (2) */
  int32_t c;              /* model.num_channels (128) */
  int32_t g;              /* growth (128) */
  int32_t bn;             /* bottleneck_factor (4) */
  int32_t num_targets;    /* 1 if training.target_instrument else len(training.instruments) */
  int32_t max_batch;
} b200sep_tfcnet_config;
int64_t b200sep_tfcnet_param_count(const b200sep_tfcnet_config* cfg);
int b200sep_tfcnet_create(b200sep_tfcnet** net, const b200sep_tfcnet_config* cfg, const float* params_host, int64_t n_params);
void b200sep_tfcnet_destroy(b200sep_tfcnet* net);
int64_t b200sep_tfcnet_device_bytes(const b200sep_tfcnet* net);
/* spec_in (B, 4, dim_t, dim_f) float32 [layout CTF] -> spec_out (B * num_targets, 4, dim_t, dim_f) [CTF] */
int b200sep_tfcnet_forward(b200sep_tfcnet* net, const float* spec_in, float* spec_out, int batch, void* stream);

/*
 * Rectangular overlap-add of the MDXC branch (architectures/mdxc_separator.py:395-402): chunks (n_chunks, channels, chunk_len)
 * placed every `hop` samples are summed, the slice [front, front + n_out) is taken and divided by `divisor` (= overlap).
 * out: (channels, n_out).
 */
int b200sep_rect_overlap_add(const float* chunks, int n_chunks, int channels, int chunk_len, int64_t hop, int64_t front, int64_t n_out,
                             float divisor, float* out, void* stream);
/* Time-sharded form (SURVEY.md section 8e, MDXC row): `chunks` holds the global chunks [first_chunk, first_chunk + n_local) only and
 * the samples [q_begin, q_end) of the (channels, n_out) output are written to out[c * out_ld + q - out_base] (a rank's own slice);
 * every chunk covering that range must be local. */
int b200sep_rect_overlap_add_range(const float* chunks, int first_chunk, int n_local, int n_chunks, int channels, int chunk_len, int64_t hop,
                                   int64_t front, int64_t n_out, int64_t q_begin, int64_t q_end, float divisor, float* out, int64_t out_ld,
                                   int64_t out_base, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Generalised STFT framing (HTDemucs._spec / _ispec, uvr_lib_v5/demucs/htdemucs.py:383-413 + spec.py:11-38): see stft.cu.
 */
int b200sep_stft_forward_ex(const b200sep_stft_plan* plan, const float* wave, int64_t batch_stride, int64_t chan_stride, int64_t valid_len,
                            int batch, int chunk_len, int frames, int frame_offset, float scale, int dim_f, int zero_bins, int layout,
                            int pad_mode /* 0 reflect (torch.stft), 1 zeros (librosa.stft pad_mode="constant") */, float* spec, void* stream);
int b200sep_stft_inverse_ex(const b200sep_stft_plan* plan, const float* spec, int batch, int frames, int dim_f, int layout, int out_len,
                            int ola_offset, int env_extra, float scale, float* wave, float* work, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * fp32 operators of the HTDemucs path (uvr_lib_v5/demucs/{htdemucs,hdemucs,demucs,transformer,apply}.py).  Each replaces the
 * ATen call named in its comment; tensors are contiguous float32 device arrays.
 *
 * conv2d_f32: nn.Conv1d / nn.Conv2d (hdemucs.py:107,113; demucs.py:147,150) and, with up_axis != 0, nn.ConvTranspose1d/2d
 *   (hdemucs.py:285) expressed as a 2-tap convolution over the coarse index q with up*Cout GEMM columns (column r*Cout+co ->
 *   output index q*up + r - trim, kept inside [0, out_len)).  x (B,Cin,H,W); w_blocked [Cin][KH*KW][ceil48(CoutCols)];
 *   y = act(conv + bias (+ add if add_before_act)) (+ add otherwise).  act: 0 none, 1 ReLU, 2 GELU(erf), 3 LeakyReLU(0.01), 4 sigmoid, 5 tanh (also gemm_f32).
 *   out_c_total != 0: y has out_c_total channels and this call fills [out_c_off, out_c_off + Cout) (a fused torch.cat; plain convs only).
 *   Tiled SIMT kernels for DH = 1 and (KH,KW,SH,SW,DW) in: (1,1,1,1,1) (3,3,1,1,1) (3,3,2,2,1) (1,3,1,1,1) (1,3,1,1,2) (8,1,4,1,1) (1,8,1,4,1) (2,1,1,1,1) (1,2,1,1,1);
 *   any other geometry (e.g. the (4,2) / (8,4) / (12,6)-dilated ASPP convolutions of VR 5.1, layers_new.py:96-98) runs on the tensor cores when it is large
 *   enough (Cin*KH*KW >= 32, Cout >= 16, >= 512 output pixels) and on a plain one-thread-per-output kernel otherwise.
 */
int b200sep_conv2d_f32(const float* x, const float* w_blocked, const float* bias, const float* add, float* y, int B, int Cin, int H, int W, int Cout,
                       int Ho, int Wo, int KH, int KW, int SH, int SW, int PH, int PW, int DH, int DW, int act, int add_before_act, int up_axis, int up,
                       int trim, int out_len, int out_c_total, int out_c_off, const void* w_packed, void* stream);
/* nn.GroupNorm(1, C), affine, optional activation (demucs.py:141,144).  Channel-first x (B, C, Fr, L): one sample per (b, fr) row
 * (Fr = 1: (B, C, L); Fr > 1: DConv on every frequency row without the permute of hdemucs.py:141-146); channel_last: x (B, L, C)
 * tokens (MyGroupNorm, transformer.py:184-193).
 * work: b200sep_groupnorm1_work_floats(...) floats of 16-byte aligned device scratch (per-CTA partial sums; keeps the call re-entrant). */
int64_t b200sep_groupnorm1_work_floats(int B, int C, int Fr, int64_t L);
int b200sep_groupnorm1_f32(const float* x, const float* gamma, const float* beta, float* y, int B, int C, int Fr, int64_t L, int act, int channel_last,
                           float* work, void* stream);
/* y = x.permute(p0,p1,p2,p3).contiguous() for a 4-D tensor (the einops rearranges around the transformer, transformer.py:532-555) */
int b200sep_permute4_f32(const float* x, float* y, int d0, int d1, int d2, int d3, int p0, int p1, int p2, int p3, void* stream);
/* F.glu(dim=1) on (B, 2C, L); with res/scale: y = res + scale[c] * glu  (LayerScale residual of DConv, demucs.py:92-93,166-168) */
int b200sep_glu_f32(const float* a, const float* res, const float* scale, float* y, int B, int C, int64_t L, void* stream);
/* nn.LayerNorm(C) on (rows, C) (transformer.py:481-482 and the layers' norm1/2/3) */
int b200sep_layernorm_f32(const float* x, const float* gamma, const float* beta, float* y, int64_t rows, int C, void* stream);
/* batched TN GEMM: C[z] = epi(alpha * A[z] (M,K; lda) @ Bw[z] (N,K; ldb)^T): + bias_n[n] + bias_m[m], act, then res + res_scale[n]*v
 * (nn.Linear / in_proj / out_proj / attention scores and values of nn.MultiheadAttention; LayerScale gamma_1/2, transformer.py:268-269) */
int b200sep_gemm_f32(const float* A, const float* Bw, float* C, int M, int N, int K, int lda, int ldb, int ldc, int batch, int64_t strideA,
                     int64_t strideB, int64_t strideC, float alpha, const float* bias_n, const float* bias_m, int act, const float* res,
                     const float* res_scale, const void* w_packed, void* stream);
/* Large conv2d_f32 / gemm_f32 calls run on the tensor cores (csrc/tc_f32.cu: fp32 operands split in-kernel into bf16 hi + lo, three
 * tcgen05 products, fp32 accumulation).  For STATIC B operands (weights) the split can be done once: w_packed (nullable) is the image
 * tc_pack_*_weights writes into a buffer of b200sep_tc_packed_floats(N, K) floats, K = the GEMM K (linear) or ceil8(Cin)*KH*KW (conv). */
int64_t b200sep_tc_packed_floats(int N, int K);
int b200sep_tc_pack_linear_weights(const float* W, int N, int K, int ldw, float* packed, void* stream);
int b200sep_tc_pack_conv_weights(const float* w_blocked, int Cin, int taps, int Cout, float* packed, void* stream);
/* Fused attention, head dimension 64: out[b, m, h*64 + d] = sum_n softmax_n(alpha <q[b, m, h], k[b, n, h]>) v[b, n, h*64 + d] with the scores kept on chip
 * (one tcgen05 kernel: Q K^T into TMEM, running softmax in registers, P V from shared memory).  q (B, Lq, .) / k (B, Lk, .) / out (B, Lq, .): batch and row
 * strides in floats, head h at columns [h*64, h*64 + 64);  v_is_kn = 0: vt = V TRANSPOSED, vt[b * vt_batch_stride + (h*64 + d) * vt_row_stride + n] (keys
 * contiguous);  v_is_kn = 1: plain V, vt[b * vt_batch_stride + n * vt_row_stride + h*64 + d].
 * Replaces gemm_f32 (scores) + softmax_rows_f32 + gemm_f32 (P V) of nn.MultiheadAttention (transformer.py:196-409). */
int b200sep_attention_f32(const float* q, const float* k, const float* vt, float* out, int B, int H, int Lq, int Lk, int head_dim, int64_t q_batch_stride,
                          int64_t q_row_stride, int64_t k_batch_stride, int64_t k_row_stride, int64_t vt_batch_stride, int64_t vt_row_stride,
                          int64_t out_batch_stride, int64_t out_row_stride, float alpha, int v_is_kn, float* work, void* stream);
/* work (nullable): b200sep_attention_work_floats(...) floats of 16-byte aligned device scratch.  With it Q / K / V are split into bf16 hi / lo tile images ONCE
 * (a small pre-pass) and the attention kernel fetches them with bulk copies; without it every CTA converts the tiles it reads (slower: each K / V tile is read
 * by all query tiles of its (batch, head)). */
int64_t b200sep_attention_work_floats(int B, int H, int Lq, int Lk);
/* in-place softmax over the first n columns of each row (row stride ld >= n; padding columns are left untouched) */
int b200sep_softmax_rows_f32(float* x, int64_t rows, int n, int64_t ld, void* stream);
/* batched C[z] = alpha * A[z] (M,K; lda) @ B[z] (K,N; ldb): the P @ V product of attention without a transposed copy of V */
int b200sep_gemm_kn_f32(const float* A, const float* B_kn, float* C, int M, int N, int K, int lda, int ldb, int ldc, int batch, int64_t strideA, int64_t strideB,
                        int64_t strideC, float alpha, void* stream);
/* op 0: out = alpha*a + beta*b (b NULL: + beta);  op 1: out = a*b;  with b = device {mean, std} (meanstd_f32):
 * op 2: out = (a - mean) / (1e-5 + std);  op 3: out = a*std + mean  (htdemucs.py:501-510, :588-589, :611-612) */
int b200sep_ew_f32(const float* a, const float* b, float* out, int64_t n, float alpha, float beta, int op, void* stream);
/* out2[0] = mean, out2[1] = unbiased std over n elements (htdemucs.py:501-510) */
int b200sep_meanstd_f32(const float* x, int64_t n, float* out2, void* stream);
/* the same for `batch` samples x + z * x_stride in two launches: out[z * out_stride + {0, 1}]; work: b200sep_meanstd_work_floats(batch) floats, 16-byte aligned */
int64_t b200sep_meanstd_work_floats(int batch);
int b200sep_meanstd_batch_f32(const float* x, int64_t n, int batch, int64_t x_stride, float* out, int out_stride, float* work, void* stream);
/* One fused DConv residual layer (uvr_lib_v5/demucs/demucs.py:85-168, `layers[d]` of DConv.forward):
 *   y = x + ls * GLU(GroupNorm(1,2C)(Conv1d(hid->2C,1)(GELU(GroupNorm(1,hid)(Conv1d(C->hid,3,dilation)(x))))))
 * on (B, C, Fr, L) with one GroupNorm sample per (b, fr) row (hdemucs.py:141-146).  w0 (hid, C, 3), w3 (2C, hid); y may alias x.
 * u_in (nullable): the (B, hid, Fr, L) output of the first convolution computed by the caller (w0 is then unused).
 * work: b200sep_dconv_work_floats(...) floats, 16-byte aligned.  See csrc/dconv_fused.cu for the three-pass scheme. */
int64_t b200sep_dconv_work_floats(int B, int C, int Fr, int64_t L, int hid);
int b200sep_dconv_f32(const float* x, float* y, const float* w0, const float* b0, const float* g1, const float* be1, const float* w3, const float* b3,
                      const float* g4, const float* be4, const float* ls, int B, int C, int Fr, int64_t L, int hid, int dilation, const float* u_in,
                      float* work, void* stream);
/* apply_model's split branch (demucs/apply.py:215-250): triangle-weighted overlap-add of segments (n_segs, channels, seg_len;
 * each already centre-trimmed to its valid length, stored from sample 0) at stride `stride` over a signal of `length` samples,
 * normalised by the summed weights.  out (channels, n_out): out[c][n] (+)= scale * chan_scale[c] * signal[c][q0 + n]
 * -- q0/scale/accumulate fold in the shift average (apply.py:197-214), chan_scale (nullable) the bag weights (apply.py:169-195). */
int b200sep_triangle_overlap_add(const float* segs, int n_segs, int channels, int seg_len, int64_t stride, int64_t length, int64_t q0, int64_t n_out,
                                 float scale, const float* chan_scale, int accumulate, float* out, void* stream);
/* Time-sharded form (SURVEY.md section 8e, Demucs row): `segs` holds the global segments [first_seg, first_seg + n_local) only; the n_out
 * samples go to out[c * out_ld + out_off + n] (a slice of full-length rows); every segment covering [q0, q0 + n_out) must be local. */
int b200sep_triangle_overlap_add_range(const float* segs, int first_seg, int n_local, int n_segs, int channels, int seg_len, int64_t stride,
                                       int64_t length, int64_t q0, int64_t n_out, float scale, const float* chan_scale, int accumulate, float* out,
                                       int64_t out_ld, int64_t out_off, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Operators of the VR path (uvr_lib_v5/vr_network/{nets,layers}.py, architectures/vr_separator.py, uvr_lib_v5/spec_utils.py).
 * Spectrograms are 4 float planes (L re, L im, R re, R im) of (bins, frames), the CFT layout of the STFT entry points.
 */
/* depthwise 3x3, dilation = padding = d: the first conv of SeperableConv2DBNActiv (layers.py:60-70); w (C, 9) */
int b200sep_dwconv3x3_f32(const float* x, const float* w, float* y, int B, int C, int H, int W, int dilation, void* stream);
/* F.interpolate(scale_factor=2, mode="bilinear", align_corners=True) (Decoder, layers.py:175) into channels [dst_c_off, +C) of (B, dst_c_total, 2H, 2W) */
int b200sep_upsample2x_bilinear_f32(const float* x, float* y, int B, int C, int H, int W, int dst_c_total, int dst_c_off, void* stream);
/* nn.AdaptiveAvgPool2d((1, None)) (ASPPModule.conv1, layers.py:232): (BC, H, W) -> (BC, W) */
int b200sep_mean_h_f32(const float* x, float* y, int BC, int H, int W, void* stream);
/* dst[i0*ds0 + i1*ds1 + i2*ds2 + i3*ds3] = src[i0*ss0 + ...] over a (d0,d1,d2,d3) index box: torch.cat / crop_center / broadcast / patch slicing */
int b200sep_copy4_f32(const float* src, float* dst, int d0, int d1, int d2, int d3, int64_t ss0, int64_t ss1, int64_t ss2, int64_t ss3, int64_t ds0,
                      int64_t ds1, int64_t ds2, int64_t ds3, void* stream);
/* x[plane][bin][t] *= gain[bin]: pre-filter of combine_spectrograms (spec_utils.py:266-277), fft_lp_filter / fft_hp_filter (:410-429) */
int b200sep_bin_gain_f32(float* x, const float* gain, int planes, int bins, int frames, void* stream);
/* |X| written at column pad_l of a zero-filled (2, bins, frames_out) buffer (spec_utils.preprocess + np.pad, vr_separator.py:345-349) */
int b200sep_vr_magnitude_pad(const float* spec, float* mag, int bins, int frames, int frames_out, int pad_l, void* stream);
/* adjust_aggr + the masked spectrograms (spec_utils.py:472-492, vr_separator.py:329-343): m = mask^e; y = m*X; v = (1-m)*X; non-finite -> 0.
 * mask (2, bins, mask_stride); e = exp_low_* below split_bin, exp_high_* from it on, per channel. */
int b200sep_vr_apply_mask(const float* mask, int mask_stride, const float* spec, int bins, int frames, int split_bin, float exp_low_left, float exp_high_left,
                          float exp_low_right, float exp_high_right, float* y_spec, float* v_spec, void* stream);
/* enable_post_process (vr_separator.py:334-335): adjust_aggr in place, the per-frame minimum merge_artifacts thresholds (spec_utils.py:187), and
 * y_mask += weight[t] * (1 - y_mask) (:213-214); the run detection between the last two is host logic on the frames-long vector */
int b200sep_vr_mask_pow(float* mask, int mask_stride, int bins, int frames, int split_bin, float exp_low_left, float exp_high_left, float exp_low_right,
                        float exp_high_right, void* stream);
int b200sep_vr_frame_min(const float* mask, int mask_stride, int rows, int frames, float* out, void* stream);
int b200sep_vr_mask_merge(float* mask, const float* frame_weight, int mask_stride, int rows, int frames, void* stream);
/* high_end_process (vr_separator.py:368-372; spec_utils.mirroring :458-463 + cmb_spectrogram_to_wave :354-356): bins [max_bin-h, max_bin) of the top band's
 * un-cropped spectrogram (4, band_bins, frames) <- the kept input high end (4, high_rows, high_frames) limited in magnitude by the flipped combined-spectrogram
 * bins [pre_filter_start-10-h, pre_filter_start-10) */
int b200sep_vr_mirror_high_end(const float* spec_m, int bins, const float* high_end, int high_rows, int high_frames, float* band_spec, int band_bins, int frames,
                               int h, int max_bin, int pre_filter_start, void* stream);
/* scipy.signal.resample_poly's upfirdn (== librosa.resample(res_type="polyphase"), vr_separator.py:280):
 * y[c][k] = sum_i x[c][i] * taps[(k + n_pre_remove)*down - i*up];  taps = the zero-padded FIR scaled by `up` */
int b200sep_resample_poly_f32(const float* x, const float* taps, int n_taps, int up, int down, int64_t n_pre_remove, int channels, int64_t n_in,
                              int64_t n_out, float* y, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Operators of the BS-Roformer path (uvr_lib_v5/roformer/bs_roformer.py, attend.py; mdxc_separator.py:272-343).
 */
/* RMSNorm (bs_roformer.py:30-37): y = F.normalize(x, dim=-1) * sqrt(C) * gamma on `rows` rows of C columns (row strides ld_in / ld_out:
 * a band of the band-split input is a column slice) */
int b200sep_rmsnorm_f32(const float* x, const float* gamma, float* y, int64_t rows, int C, int64_t ld_in, int64_t ld_out, void* stream);
/* "b n (qkv h d) -> qkv b h n d" + rotary_embed.rotate_queries_or_keys on q and k (bs_roformer.py:67-72; rotary-embedding-torch defaults):
 * qkv (B, n, 3*H*dh) -> q, k, v (B, H, n, dh) */
int b200sep_rope_split_heads_f32(const float* qkv, const float* freqs, float* q, float* k, float* v, int B, int n, int H, int dh, void* stream);
/* out * sigmoid(gates) + "b h n d -> b n (h d)" (bs_roformer.py:76-81): o (B, H, n, dh), gates (B*n, H) -> y (B*n, H*dh) */
int b200sep_gate_merge_heads_f32(const float* o, const float* gates, float* y, int B, int n, int H, int dh, void* stream);
/* nn.GLU(dim=-1) of MaskEstimator (bs_roformer.py:175): a (rows, 2C; ld_in) -> y (rows, C; ld_out) */
int b200sep_glu_rows_f32(const float* a, float* y, int64_t rows, int C, int64_t ld_in, int64_t ld_out, void* stream);
/* stft_repr * mask as complex numbers and the re-ordering to iSTFT planes (bs_roformer.py:472-484):
 * stft_tf (B, T, F, 4) and mask (B, n_stems, T, F, 4) with feature order (f, s, c) -> planes (B*n_stems, 4, F, T) [L re, L im, R re, R im] */
int b200sep_roformer_mask_apply(const float* stft_tf, const float* mask, float* planes, int B, int n_stems, int T, int F, void* stream);
/* Mel-Band Roformer: stft_repr[batch_arange, freq_indices] (mel_band_roformer.py:300-303) on (re, im) pairs: dst[row][g] = src[row][idx[g]] */
int b200sep_gather_pairs_f32(const float* src, const int* idx, float* dst, int64_t rows, int n_src_pairs, int n_gather, void* stream);
/* masks.scatter_add_ / num_bands_per_freq (mel_band_roformer.py:306-318) as an output-side gather: out[row][fs] = mean of mask_gathered[row][pos] over
 * pos in csr_positions[csr_offsets[fs] .. csr_offsets[fs+1])  (complex pairs) */
int b200sep_mask_average_f32(const float* mask_gathered, const int* csr_offsets, const int* csr_positions, float* mask_out, int64_t rows, int n_gather, int n_out,
                             void* stream);
/* Roformer branch of MDXCSeparator.demix (mdxc_separator.py:310-343): out[c][q] = sum_i window[q - starts[i]] * chunks[i][c][q - starts[i]] /
 * max(sum_i window[q - starts[i]], 1e-10); chunks (n_chunks, channels, len), starts device int64[n_chunks], non-decreasing */
int b200sep_overlap_add_starts(const float* chunks, const int64_t* starts, const float* window, int n_chunks, int channels, int len, int64_t n_out, float* out,
                               void* stream);
/* Time-sharded form: `chunks` (n_local, channels, len) holds the global chunks [first, first + n_local) only, `starts` is the whole global list, and the
 * samples [q_begin, q_end) of the (channels, n_out) output are written to out[c * out_ld + q - out_base].  Every chunk covering that range must be
 * local (B200SEP_ERR_ARG otherwise); when the run is not the whole list, checking this reads two entries of `starts` back and synchronises `stream`.
 * Each sample gets the same contributions in the same order as from b200sep_overlap_add_starts, so a slice is bit-identical to the full call's columns. */
int b200sep_overlap_add_starts_range(const float* chunks, const int64_t* starts, const float* window, int first, int n_local, int n_chunks, int channels, int len,
                                     int64_t n_out, int64_t q_begin, int64_t q_end, float* out, int64_t out_ld, int64_t out_base, void* stream);

/* nn.LSTM(bidirectional=True), one layer (LSTMModule of VR 5.1, layers_new.py:124-149): the recurrence only.  x_proj (2, T, N, 4*hid) = the input
 * projections x_t @ W_ih^T + b_ih + b_hh of the forward / reverse direction (gate order i, f, g, o; computed with gemm_f32), w_hh (2, 4*hid, hid);
 * out (T, N, 2*hid) = [forward h_t | reverse h_t].  hid <= 96. */
int b200sep_lstm_bidir_f32(const float* x_proj, const float* w_hh, float* out, int T, int N, int hid, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Hybrid Demucs v3 (uvr_lib_v5/demucs/hdemucs.py, demucs.py): the operators its DConv branches add to the HTDemucs set.
 * groupnorm_f32: nn.GroupNorm(groups, C) (hdemucs.py:87-88, norm_groups = 4) on contiguous channel-first x (B, C, X), affine, optional activation.
 * lstm_bidir_wide_f32: the recurrence of one bidirectional nn.LSTM layer for ANY hidden size (BLSTM of DConv, demucs.py:26-30: hid = 192 / 384 in
 *   the released models).  Same x_proj (2, T, N, 4*hid) / out (T, N, 2*hid) as lstm_bidir_f32; the recurrent matrix is passed TRANSPOSED,
 *   w_hh_t (2, hid, 4*hid).  A thread-block cluster splits the hidden units and exchanges h_t through distributed shared memory.
 * lstm_frames_gather_f32 / _scatter_f32: BLSTM.forward's framing (demucs.py:38-45 unfold into frames of `width` every `stride`; :52-64 the
 *   trimmed concatenation back + the skip connection): x (B, C, T) -> frames (width, B*n_frames, C);  frames -> y (B, C, T) = skip + kept parts.
 *   n_frames = 1, width = T is the unframed case (a pure permute).
 * local_state_attn_f32: LocalState.forward (demucs.py:197-231, nfreqs = 0) between the 1x1 projections: query / key / content (B, C, T),
 *   decay (B, heads*ndecay, T) = the query_decay convolution BEFORE the sigmoid -> out (B, C, T) = attention-weighted content
 *   (decay penalty, -100 on the diagonal, softmax over the key axis).  C / heads in {1,2,3,4,6,8,12,16,24,32,48,64,96}.
 * add_rowvec_f32: x (B, R, L) += v (R) broadcast over B and L: the frequency embedding after the first encoder (hdemucs.py:708-713), R = C * Fr. */
int b200sep_add_rowvec_f32(float* x, const float* v, int B, int R, int64_t L, void* stream);
int64_t b200sep_groupnorm_work_floats(int B, int C, int groups, int64_t X);
int b200sep_groupnorm_f32(const float* x, const float* gamma, const float* beta, float* y, int B, int C, int groups, int64_t X, int act, float* work, void* stream);
int b200sep_lstm_bidir_wide_f32(const float* x_proj, const float* w_hh_t, float* out, int T, int N, int hid, void* stream);
int b200sep_lstm_frames_gather_f32(const float* x, float* frames, int B, int C, int T, int n_frames, int width, int stride, void* stream);
int b200sep_lstm_frames_scatter_f32(const float* frames, const float* skip, float* y, int B, int C, int T, int n_frames, int width, int stride, void* stream);
int b200sep_local_state_attn_f32(const float* query, const float* key, const float* content, const float* decay, float* out, int B, int C, int T, int heads,
                                 int ndecay, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Ensembling of several models' stems (audio_separator/separator/ensembler.py:10-156, spec_utils.ensembling :583-608).
 * ensemble_f32: x (n_models, n) -> out (n); algo 0 weighted mean (weights: device float[n_models]), 1 median, 2 / 3 the value of smallest / largest
 * magnitude (first on ties): avg_wave, median_wave, min_wave, max_wave, and avg_fft / median_fft applied to spectrogram planes.
 * ensemble_spec_abs: planes (n_models, 4, plane_elems) -> (4, plane_elems), per complex entry the model with the smallest / largest modulus
 * (last_wins 0: min_fft / max_fft; 1: uvr_min_spec / uvr_max_spec).  n_models <= 16. */
int b200sep_ensemble_f32(const float* x, int n_models, int64_t n, const float* weights, int algo, float* out, void* stream);
int b200sep_ensemble_spec_abs(const float* planes, int n_models, int64_t plane_elems, int take_max, int last_wins, float* out, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * Self-tests of the tensor-core ("bf16x3 pair") operators in isolation: fp32 device tensors in, the operator runs
 * exactly as inside the network (split into bf16 hi/lo planes -> tcgen05 kernel -> join), fp32 out.  Synchronous.
 *   gemm   : out[M][N] = act((a[M][K] @ w[N][K]^T) * scale[c] + shift[c]) (+ res),  c = (row / rows_per_channel) % channels
 *   conv3x3: out(B,Cout,T,F) = act(conv2d(x(B,Cin,T,F), w(Cout,Cin,3,3), padding=1) * scale[co] + shift[co]);  w is a HOST pointer
 */
int b200sep_selftest_umma_gemm(const float* a, const float* w, const float* res, float* out, int M, int N, int K, int rows_per_channel,
                               int channels, const float* scale, const float* shift, int relu, void* stream);
int b200sep_selftest_umma_conv3x3(const float* x, const float* w_host, float* out, int B, int Cin, int Cout, int T, int F, const float* scale,
                                  const float* shift, int relu, void* stream);
/*   updown : up != 0: out(B,Cout,2T,2F) = act(conv_transpose2d(x, w(Cin,Cout,2,2), stride=2) * scale + shift) [* skip(B,Cout,2T,2F)]
 *            up == 0: out(B,Cout,T/2,F/2) = act(conv2d(x, w(Cout,Cin,2,2), stride=2) * scale + shift);  w is a HOST pointer, skip may be NULL */
int b200sep_selftest_umma_updown(const float* x, const float* w_host, const float* skip, float* out, int B, int Cin, int Cout, int T, int F,
                                 const float* scale, const float* shift, int relu, int up, void* stream);
/*   ex     : the epilogue options MDX23C uses.  kind 0 conv3x3, 1 pw (1x1), 2 down (2x2 s2), 3 up (2x2 transposed s2); w_host as above
 *            ((Cout,Cin,3,3) / (Cout,Cin) / (Cout,Cin,2,2) / (Cin,Cout,2,2)).  y = act(op(x)) (act 0 none, 1 ReLU, 2 GELU); then y += res
 *            (conv3x3, pw) or y *= res (up); then y *= mul (conv3x3, pw); res and mul are (B, Cout, T', F') and may be NULL.  y goes to channels
 *            [out_c_off, out_c_off + Cout) of out (B, out_c_total, T', F') (out_c_total 0 = Cout), as a pair, or as plain fp32 when out_f32 != 0 (pw only).
 *            `out` is read first and split into the pair buffer, so channels outside the slice round-trip. */
int b200sep_selftest_umma_ex(int kind, const float* x, const float* w_host, const float* res, const float* mul, float* out, int B, int Cin, int Cout,
                             int T, int F, int act, int out_c_total, int out_c_off, int out_f32, void* stream);
/*   instnorm_act: out (B, C, P) = act(instance_norm(channels [x_c_off, x_c_off + C) of x (B, x_c_total, P); gamma, beta, eps 1e-5)), act 0 / 1 ReLU / 2 GELU;
 *            gamma / beta are device pointers, P % 8 == 0 */
int b200sep_selftest_instnorm_act(const float* x, const float* gamma, const float* beta, float* out, int B, int C, int x_c_total, int x_c_off, int64_t P,
                                  int act, void* stream);

/* ---------------------------------------------------------------------------------------------------
 * CUDA-graph capture of a launch list issued through this ABI (csrc/api.cu): bracket any sequence of operator calls on `stream`, replay it with
 * one launch.  The buffers must keep their addresses; run the sequence once before capturing.
 */
typedef struct b200sep_graph b200sep_graph;
int b200sep_capture_begin(void* stream);
int b200sep_capture_end(void* stream, b200sep_graph** out);
int b200sep_graph_launch(b200sep_graph* graph, void* stream);
void b200sep_graph_destroy(b200sep_graph* graph);

#ifdef __cplusplus
}
#endif
#endif /* B200SEP_H */
