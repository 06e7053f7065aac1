"""BS-Roformer on the operator kernels of libb200sep.so.

BSRoformerNet.forward replaces BSRoformer.forward (uvr_lib_v5/roformer/bs_roformer.py:418-497) and RoformerEngine the Roformer branch of
MDXCSeparator.demix (architectures/mdxc_separator.py:272-343).  Launch order only: STFT -> band split (RMSNorm + Linear per band) ->
depth x [time transformer over (b f) sequences, frequency transformer over (b t) sequences] (RMSNorm, fused QKV GEMM, rotary + head split,
QK^T / softmax / PV GEMMs, sigmoid gates + head merge, output GEMM with residual, RMSNorm + GELU MLP with residual) -> final RMSNorm ->
per-band mask MLPs (tanh, GLU) -> complex mask product -> iSTFT -> Hamming overlap-add with weight counter.
All GEMMs run through b200sep_gemm_f32 (tensor cores for the large ones, static weights pre-split once).
Covered: BS-Roformer (linear_transformer_depth = 0) and Mel-Band Roformer, stereo, any num_stems / mask_estimator_depth / band layout; mono is not.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np
import torch

from ._lib import LAYOUT_CFT, check, lib
from .demucs import _FUSED_ATTENTION, ACT_GELU, ACT_NONE, _new, _packed_linear
from .engine import StftPlan, _ptr, _require_cuda, _stream

ACT_TANH = 5
DEFAULT_FREQS_PER_BANDS = (2,) * 24 + (4,) * 12 + (12,) * 8 + (24,) * 8 + (48,) * 8 + (128, 129)


@dataclass
class BSRoformerConfig:
    """BSRoformer constructor arguments that shape the graph (bs_roformer.py:300-345)."""

    dim: int = 512
    depth: int = 12
    stereo: bool = True
    num_stems: int = 1
    time_transformer_depth: int = 1
    freq_transformer_depth: int = 1
    linear_transformer_depth: int = 0
    freqs_per_bands: tuple = DEFAULT_FREQS_PER_BANDS
    dim_head: int = 64
    heads: int = 8
    mlp_expansion_factor: int = 4
    mask_estimator_depth: int = 2
    stft_n_fft: int = 2048
    stft_hop_length: int = 512
    stft_win_length: int = 2048
    stft_normalized: bool = False

    @classmethod
    def from_model_section(cls, m: dict) -> "BSRoformerConfig":
        known = {k: m[k] for k in cls.__dataclass_fields__ if k in m}
        if "freqs_per_bands" in known:
            known["freqs_per_bands"] = tuple(known["freqs_per_bands"])
        cfg = cls(**known)
        if m.get("linear_transformer_depth", 0) or m.get("sage_attention", False):
            raise NotImplementedError("linear-attention / sage-attention Roformer variants are not covered")
        if m.get("stft_window_fn") not in (None, "torch.hann_window"):
            raise NotImplementedError("only the Hann STFT window is covered")
        if cfg.stft_normalized or cfg.stft_win_length != cfg.stft_n_fft:
            raise NotImplementedError("stft_normalized / win_length != n_fft are not covered")
        if sum(cfg.freqs_per_bands) != cfg.stft_n_fft // 2 + 1:
            raise ValueError("the number of freqs in the bands must equal n_fft/2 + 1")
        return cfg

    @property
    def audio_channels(self):
        return 2 if self.stereo else 1

    @property
    def band_dims(self):
        return tuple(2 * f * self.audio_channels for f in self.freqs_per_bands)


@dataclass
class MelBandRoformerConfig:
    """MelBandRoformer constructor arguments that shape the graph (mel_band_roformer.py:124-160)."""

    dim: int = 384
    depth: int = 6
    stereo: bool = True
    num_stems: int = 1
    time_transformer_depth: int = 1
    freq_transformer_depth: int = 1
    num_bands: int = 60
    dim_head: int = 64
    heads: int = 8
    mask_estimator_depth: int = 1
    sample_rate: int = 44100
    stft_n_fft: int = 2048
    stft_hop_length: int = 512
    stft_win_length: int = 2048
    stft_normalized: bool = False

    @classmethod
    def from_model_section(cls, m: dict) -> "MelBandRoformerConfig":
        cfg = cls(**{k: m[k] for k in cls.__dataclass_fields__ if k in m})
        if m.get("sage_attention", False) or m.get("match_input_audio_length", False):
            raise NotImplementedError("sage_attention / match_input_audio_length are not covered")
        if m.get("stft_window_fn") not in (None, "torch.hann_window"):
            raise NotImplementedError("only the Hann STFT window is covered")
        if cfg.stft_normalized or cfg.stft_win_length != cfg.stft_n_fft:
            raise NotImplementedError("stft_normalized / win_length != n_fft are not covered")
        return cfg

    @property
    def audio_channels(self):
        return 2 if self.stereo else 1

    @property
    def freqs_per_bands(self):
        return tuple(int(v) for v in mel_band_layout(self)[2])

    @property
    def band_dims(self):
        return tuple(2 * f * self.audio_channels for f in self.freqs_per_bands)


def _slaney_mel(f):
    f = np.asarray(f, dtype=np.float64)
    lin = f * 3.0 / 200.0
    return np.where(f >= 1000.0, 15.0 + np.log(np.maximum(f, 1e-300) / 1000.0) / (np.log(6.4) / 27.0), lin)


def _slaney_hz(m):
    m = np.asarray(m, dtype=np.float64)
    return np.where(m >= 15.0, 1000.0 * np.exp((np.log(6.4) / 27.0) * (m - 15.0)), m * 200.0 / 3.0)


def mel_band_layout(cfg: "MelBandRoformerConfig"):
    """Which STFT bins each band covers: the support of librosa.filters.mel(sr, n_fft, n_mels=num_bands) (Slaney scale, triangles between
    consecutive mel points; bin 0 forced into the first band and the last bin into the last one), as MelBandRoformer.__init__ derives it
    (mel_band_roformer.py:239-262).  -> (mask (bands, F), gather indices over the (f s) axis, freqs per band, bands per freq)"""
    n_f = cfg.stft_n_fft // 2 + 1
    fft_f = np.fft.rfftfreq(n=cfg.stft_n_fft, d=1.0 / cfg.sample_rate)
    pts = _slaney_hz(np.linspace(_slaney_mel(0.0), _slaney_mel(cfg.sample_rate / 2.0), cfg.num_bands + 2))
    widths = np.diff(pts)
    ramps = np.subtract.outer(pts, fft_f)
    tri = np.zeros((cfg.num_bands, n_f), dtype=np.float32)
    for i in range(cfg.num_bands):
        tri[i] = np.maximum(0, np.minimum(-ramps[i] / widths[i], ramps[i + 2] / widths[i + 1]))
    tri *= (2.0 / (pts[2 : cfg.num_bands + 2] - pts[: cfg.num_bands]))[:, None]
    tri[0, 0] = 1.0
    tri[-1, -1] = 1.0
    mask = tri > 0
    if not mask.any(axis=0).all():
        raise ValueError("all frequencies need to be covered by all bands for now")
    idx = np.tile(np.arange(n_f), (cfg.num_bands, 1))[mask]
    if cfg.stereo:
        idx = (idx[:, None] * 2 + np.arange(2)[None, :]).reshape(-1)
    return mask, idx.astype(np.int64), mask.sum(1), mask.sum(0)


def gemm(a_ptr, w, c_ptr, M, lda, ldc, bias=None, act=ACT_NONE, res_ptr=None):
    """rows x K (row stride lda) @ w (N, K)^T + bias -> rows x N at row stride ldc (+ res with the same strides)."""
    N, K = w.shape
    pk = _packed_linear(w)
    check(lib.b200sep_gemm_f32(a_ptr, _ptr(w), c_ptr, M, N, K, lda, K, ldc, 1, 0, 0, 0, 1.0, _ptr(bias) if bias is not None else None, None, act, res_ptr, None,
                               _ptr(pk) if pk is not None else None, _stream()), "gemm_f32")


def rmsnorm(x, gamma, rows, C, ld_in=None, out=None):
    y = out if out is not None else _new((rows, C), x)
    check(lib.b200sep_rmsnorm_f32(x.data_ptr() if isinstance(x, torch.Tensor) else x, _ptr(gamma), _ptr(y), rows, C, ld_in or C, C, _stream()), "rmsnorm_f32")
    return y


class BSRoformerNet:
    """BS-Roformer (cfg: BSRoformerConfig) or Mel-Band Roformer (cfg: MelBandRoformerConfig): the graphs differ only in the band layout (disjoint
    slices vs gathered, overlapping mel bands whose masks are averaged), the per-transformer output norm and the mask MLP depth."""

    def __init__(self, cfg, state: dict, device=None):
        _require_cuda()
        self.cfg = cfg
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())  # one process per GPU: the rank's own device
        if not cfg.stereo:
            raise NotImplementedError("mono BS-Roformer checkpoints are not covered (the STFT kernels process stereo pairs)")
        self.stft = StftPlan(cfg.stft_n_fft, cfg.stft_hop_length)
        self.W = {}
        for k, v in state.items():
            a = np.asarray(v, dtype=np.float32) if not isinstance(v, torch.Tensor) else v.detach().to(torch.float32).numpy()
            self.W[k] = torch.from_numpy(np.ascontiguousarray(a)).to(self.device)
        for n in ("band_split.to_features.0.1.weight", "layers.0.0.layers.0.0.to_qkv.weight", "mask_estimators.0.to_freqs.0.0.0.weight"):
            if n not in self.W:
                raise ValueError(f"state dict lacks {n}: not a Roformer checkpoint")
        if self.W["layers.0.0.layers.0.0.to_qkv.weight"].shape != (3 * cfg.heads * cfg.dim_head, cfg.dim):
            raise ValueError("dim / heads / dim_head do not match the checkpoint")
        self.band_dims = cfg.band_dims
        if f"band_split.to_features.{len(self.band_dims) - 1}.1.weight" not in self.W or f"band_split.to_features.{len(self.band_dims)}.1.weight" in self.W:
            raise ValueError("the band layout does not match the checkpoint")
        for bi, d_in in enumerate(self.band_dims):
            if self.W[f"band_split.to_features.{bi}.1.weight"].shape[1] != d_in:
                raise ValueError(f"band {bi}: the checkpoint expects {self.W[f'band_split.to_features.{bi}.1.weight'].shape[1]} inputs, the band layout gives {d_in}")
        self.n_mask_linear = sum(1 for k in self.W if k.startswith("mask_estimators.0.to_freqs.0.0.") and k.endswith(".weight"))
        self.mel = isinstance(cfg, MelBandRoformerConfig)
        if self.mel:  # overlapping bands: gather indices for the band split, CSR lists for the mask average
            _, idx, _, _ = mel_band_layout(cfg)
            FS = (cfg.stft_n_fft // 2 + 1) * 2
            order = np.argsort(idx, kind="stable")
            counts = np.bincount(idx, minlength=FS)
            self.gather_idx = torch.from_numpy(idx.astype(np.int32)).to(self.device)
            self.csr_off = torch.from_numpy(np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)).to(self.device)
            self.csr_pos = torch.from_numpy(order.astype(np.int32)).to(self.device)

    # ---- one Transformer (norm_output=False): x (Bq, n, d) in place
    def _transformer(self, x, Bq, n, p, depth):
        cfg, W = self.cfg, self.W
        d, H, dh = cfg.dim, cfg.heads, cfg.dim_head
        inner = H * dh
        rows = Bq * n
        ldv = -(-n // 4) * 4  # row stride of the score matrix: a 16-byte aligned K-major A operand for the P@V GEMM
        for l in range(depth):
            a, f = f"{p}.layers.{l}.0", f"{p}.layers.{l}.1"
            xn = rmsnorm(x, W[f"{a}.norm.gamma"], rows, d)
            qkv = _new((rows, 3 * inner), x)
            gemm(_ptr(xn), W[f"{a}.to_qkv.weight"], _ptr(qkv), rows, d, 3 * inner)
            q, k, v = _new((Bq, H, n, dh), x), _new((Bq, H, n, dh), x), _new((Bq, H, n, dh), x)
            check(lib.b200sep_rope_split_heads_f32(_ptr(qkv), _ptr(W[f"{a}.rotary_embed.freqs"]), _ptr(q), _ptr(k), _ptr(v), Bq, n, H, dh, _stream()), "rope_split_heads_f32")
            o = _new((Bq, H, n, dh), x)
            if dh == 64 and _FUSED_ATTENTION:  # scores stay on chip (b200sep_attention_f32): every (batch, head) pair is one batch entry of the kernel, V untransposed
                work = _new((lib.b200sep_attention_work_floats(Bq * H, 1, n, n),), x)
                check(lib.b200sep_attention_f32(_ptr(q), _ptr(k), _ptr(v), _ptr(o), Bq * H, 1, n, n, dh, n * dh, dh, n * dh, dh, n * dh, dh, n * dh, dh, dh**-0.5, 1,
                                                _ptr(work), _stream()), "attention_f32")
            else:
                sc = _new((Bq * H, n, ldv), x)  # padding columns n..ldv-1 are never read: the P@V GEMM runs K = n over rows of stride ldv
                check(lib.b200sep_gemm_f32(_ptr(q), _ptr(k), _ptr(sc), n, n, dh, dh, dh, ldv, Bq * H, n * dh, n * dh, n * ldv, dh**-0.5, None, None, 0, None, None, None,
                                           _stream()), "gemm_f32(scores)")
                check(lib.b200sep_softmax_rows_f32(_ptr(sc), Bq * H * n, n, ldv, _stream()), "softmax_rows_f32")
                check(lib.b200sep_gemm_kn_f32(_ptr(sc), _ptr(v), _ptr(o), n, dh, n, ldv, dh, dh, Bq * H, n * ldv, n * dh, n * dh, 1.0, _stream()), "gemm_kn_f32(PV)")
            gates = _new((rows, H), x)
            gemm(_ptr(xn), W[f"{a}.to_gates.weight"], _ptr(gates), rows, d, H, bias=W[f"{a}.to_gates.bias"])
            merged = _new((rows, inner), x)
            check(lib.b200sep_gate_merge_heads_f32(_ptr(o), _ptr(gates), _ptr(merged), Bq, n, H, dh, _stream()), "gate_merge_heads_f32")
            x2 = _new((rows, d), x)
            gemm(_ptr(merged), W[f"{a}.to_out.0.weight"], _ptr(x2), rows, inner, d, res_ptr=_ptr(x))  # attn(x) + x
            hn = rmsnorm(x2, W[f"{f}.net.0.gamma"], rows, d)
            hid = W[f"{f}.net.1.bias"].numel()
            h = _new((rows, hid), x)
            gemm(_ptr(hn), W[f"{f}.net.1.weight"], _ptr(h), rows, d, hid, bias=W[f"{f}.net.1.bias"], act=ACT_GELU)
            x = _new((rows, d), x)
            gemm(_ptr(h), W[f"{f}.net.4.weight"], _ptr(x), rows, hid, d, bias=W[f"{f}.net.4.bias"], res_ptr=_ptr(x2))  # ff(x) + x
        if f"{p}.norm.gamma" in W:  # Transformer(norm_output=True): the Mel-Band variant (mel_band_roformer.py:82-101)
            x = rmsnorm(x, W[f"{p}.norm.gamma"], rows, d)
        return x

    def forward(self, raw_audio: torch.Tensor) -> torch.Tensor:
        """(b, 2, L) float32 cuda -> (b, 2, L') for num_stems == 1, else (b, n, 2, L'), L' = hop * (L // hop)."""
        cfg, W = self.cfg, self.W
        assert raw_audio.dim() == 3 and raw_audio.shape[1] == 2 and raw_audio.dtype == torch.float32 and raw_audio.is_cuda
        b, _, L = raw_audio.shape
        d, nb, S = cfg.dim, len(self.band_dims), cfg.num_stems
        Fq = cfg.stft_n_fft // 2 + 1
        spec = self.stft.forward(raw_audio, Fq, 0, LAYOUT_CFT)  # torch.stft(center=True, reflect, hann): planes (b, 4, F, T)
        T = spec.shape[3]
        feat = _new((b, T, Fq, 4), spec)  # "b s f t c -> b t (f s c)": feature index (f, s, c)
        check(lib.b200sep_permute4_f32(_ptr(spec), _ptr(feat), b, 4, Fq, T, 0, 3, 2, 1, _stream()), "permute4_f32")
        rows = b * T
        src = feat
        if self.mel:  # stft_repr[batch_arange, freq_indices]: every band gets its own copy of the (freq, channel) pairs it covers
            G = self.gather_idx.numel()
            src = _new((b, T, G, 2), spec)
            check(lib.b200sep_gather_pairs_f32(_ptr(feat), _ptr(self.gather_idx), _ptr(src), rows, Fq * 2, G, _stream()), "gather_pairs_f32")
        nfeat = src.shape[2] * src.shape[3] if self.mel else Fq * 4
        x = _new((b, T, nb, d), spec)
        off = 0
        for bi, d_in in enumerate(self.band_dims):  # BandSplit (bs_roformer.py:134-150)
            xn = rmsnorm(src.data_ptr() + off * 4, W[f"band_split.to_features.{bi}.0.gamma"], rows, d_in, ld_in=nfeat, out=_new((rows, d_in), spec))
            gemm(_ptr(xn), W[f"band_split.to_features.{bi}.1.weight"], x.data_ptr() + bi * d * 4, rows, d_in, nb * d, bias=W[f"band_split.to_features.{bi}.1.bias"])
            off += d_in
        for i in range(cfg.depth):
            xt = _new((b, nb, T, d), x)  # "b t f d -> (b f) t d"
            check(lib.b200sep_permute4_f32(_ptr(x), _ptr(xt), b, T, nb, d, 0, 2, 1, 3, _stream()), "permute4_f32")
            xt = self._transformer(xt.view(b * nb * T, d), b * nb, T, f"layers.{i}.0", cfg.time_transformer_depth)
            x = _new((b, T, nb, d), xt)  # "(b f) t d -> (b t) f d"
            check(lib.b200sep_permute4_f32(_ptr(xt), _ptr(x), b, nb, T, d, 0, 2, 1, 3, _stream()), "permute4_f32")
            x = self._transformer(x.view(b * T * nb, d), b * T, nb, f"layers.{i}.1", cfg.freq_transformer_depth).view(b, T, nb, d)
        xf = rmsnorm(x, W["final_norm.gamma"], rows * nb, d) if "final_norm.gamma" in W else x
        mask = _new((b, S, T, nfeat), spec)
        for si in range(S):  # MaskEstimator (bs_roformer.py:165-190)
            off = 0
            for bi, d_in in enumerate(self.band_dims):
                h_ptr, lda, kdim = xf.data_ptr() + bi * d * 4, nb * d, d
                for li in range(self.n_mask_linear):  # BS: mask_estimator_depth linears, Mel-Band: depth + 1 (their MLP helpers differ)
                    p = f"mask_estimators.{si}.to_freqs.{bi}.0.{2 * li}"
                    w = W[f"{p}.weight"]
                    last = li == self.n_mask_linear - 1
                    y = _new((rows, w.shape[0]), spec)
                    gemm(h_ptr, w, _ptr(y), rows, lda, w.shape[0], bias=W[f"{p}.bias"], act=ACT_NONE if last else ACT_TANH)
                    hold = y  # keeps the buffer alive while its raw pointer is in use
                    h_ptr, lda = _ptr(y), w.shape[0]
                for bb in range(b):  # the mask tensor is (b, S, T, features): one row block per batch element
                    check(lib.b200sep_glu_rows_f32(hold.data_ptr() + bb * T * 2 * d_in * 4, mask.data_ptr() + (((bb * S + si) * T) * nfeat + off) * 4, T, d_in, 2 * d_in, nfeat,
                                                   _stream()), "glu_rows_f32")
                off += d_in
        if self.mel:  # masks_summed / num_bands_per_freq (mel_band_roformer.py:306-318)
            full = _new((b, S, T, Fq * 4), spec)
            check(lib.b200sep_mask_average_f32(_ptr(mask), _ptr(self.csr_off), _ptr(self.csr_pos), _ptr(full), b * S * T, nfeat // 2, Fq * 2, _stream()), "mask_average_f32")
            mask = full
        planes = _new((b * S, 4, Fq, T), spec)
        check(lib.b200sep_roformer_mask_apply(_ptr(feat), _ptr(mask), _ptr(planes), b, S, T, Fq, _stream()), "roformer_mask_apply")
        wave = self.stft.inverse(planes, LAYOUT_CFT)  # torch.istft(center=True, hann): (b*S, 2, hop*(T-1))
        return wave.view(b, 2, -1) if S == 1 else wave.view(b, S, 2, -1)

    __call__ = forward


class RoformerEngine:
    """Roformer branch of MDXCSeparator.demix (mdxc_separator.py:272-343) with `batch_size` chunks per forward.

    With `dist` (torch.distributed, nccl, one process per GPU) the chunk list is time-sharded (b200/sharded.py, plan_start_shards): rank r finalises the
    output samples [N*r/W, N*(r+1)/W), computes the chunks that start there and receives from its left neighbour the chunks that reach into its range."""

    def __init__(self, net: BSRoformerNet, dim_t: int, overlap, sample_rate=44100, n_instruments=1, batch_size=1, dist=None, group=None):
        from .sharded import ShardRunner

        self.net = net
        cfg = net.cfg
        self.chunk_size = int(cfg.stft_hop_length) * (int(dim_t) - 1)  # :301
        desired = int(overlap * sample_rate)
        self.step = self.chunk_size if desired <= 0 else min(desired, self.chunk_size)  # :308-309
        self.n_instruments = int(n_instruments)
        self.batch_size = max(1, int(batch_size))
        self.device = net.device
        m = np.arange(self.chunk_size, dtype=np.float64)
        ham = 0.54 - 0.46 * np.cos(2.0 * np.pi * m / (self.chunk_size - 1)) if self.chunk_size > 1 else np.ones(1)  # scipy.signal.windows.hamming (symmetric)
        self.window = torch.from_numpy(ham.astype(np.float32)).to(self.device)
        from .graphs import GraphedForward

        self.graphed = GraphedForward(self.net.forward)
        self.runner = ShardRunner(dist, group)
        self.rank, self.world = self.runner.rank, self.runner.world

    def chunk_starts(self, N: int) -> list[int]:
        """The chunk grid of a (2, N) track (:310-315): every `step` samples, the tail clamped to N - chunk (repeated when step < chunk)."""
        C = self.chunk_size
        if N < C:
            raise NotImplementedError(f"tracks shorter than one chunk ({C} samples) are not covered by the accelerated Roformer path")
        return [i if i + C <= N else N - C for i in range(0, N, self.step)]

    def _forward_into(self, mix: torch.Tensor, starts, out: torch.Tensor, slot0: int):
        """One forward over the chunks mix[:, s : s + chunk] for s in `starts` -> out[slot0 : slot0 + len(starts)] as (S*2, chunk) rows."""
        C, S, n = self.chunk_size, self.net.cfg.num_stems, len(starts)
        batch = _new((n, 2, C), mix)
        for j, s in enumerate(starts):
            batch[j].copy_(mix[:, s : s + C])
        y = self.graphed(batch)  # (n, 2, L') or (n, S, 2, L'): CUDA-graph replay of the forward's launch list
        if y.shape[-1] != C:  # safe_len = min(length, x.shape[-1], window) (:252): hop does not divide the chunk -> zero weight beyond the model output
            raise NotImplementedError("chunk sizes that are not a multiple of the STFT hop are not covered")
        out[slot0 : slot0 + n].copy_(y.reshape(n, S * 2, C))

    def demix_device(self, mix: torch.Tensor) -> torch.Tensor:
        """mix (2, N) cuda -> (n_out, 2, N): n_out = num_stems rows for multi-stem models, 1 row for single-target models.  With `dist`: this rank's
        (n_out, 2, q1 - q0) slice of it (gather() assembles the whole on rank 0)."""
        N = mix.shape[1]
        C = self.chunk_size
        starts = self.chunk_starts(N)
        S = self.net.cfg.num_stems
        sd = torch.tensor(starts, dtype=torch.int64, device=mix.device)
        if self.runner.dist is None:
            chunks = _new((len(starts), S * 2, C), mix)
            for i0 in range(0, len(starts), self.batch_size):
                self._forward_into(mix, starts[i0 : i0 + self.batch_size], chunks, i0)
            out = _new((S * 2, N), mix)
            check(lib.b200sep_overlap_add_starts(_ptr(chunks), _ptr(sd), _ptr(self.window), len(starts), S * 2, C, N, _ptr(out), _stream()), "overlap_add_starts")
            return out.view(S, 2, N)
        from .sharded import plan_start_shards

        sh = plan_start_shards(N, self.world, starts, C)[self.rank]
        local = _new((sh.halo + sh.n_own, S * 2, C), mix)  # [halo | own]
        self.runner.wait_all(self.runner.run_units(sh, local, lambda buf, slot0, unit0, n: self._forward_into(mix, starts[unit0 : unit0 + n], buf, slot0), self.batch_size))
        n_q = sh.q1 - sh.q0
        out = _new((S * 2, n_q), mix)
        if n_q:
            check(lib.b200sep_overlap_add_starts_range(_ptr(local), _ptr(sd), _ptr(self.window), sh.c0 - sh.halo, sh.halo + sh.n_own, len(starts), S * 2, C, N, sh.q0, sh.q1,
                                                       _ptr(out), n_q, sh.q0, _stream()), "overlap_add_starts_range")
        return out.view(S, 2, n_q)

    def gather(self, part: torch.Tensor, N: int):
        """Rank 0: the full (S, 2, N) stems from every rank's demix_device slice (None elsewhere); identity on a single GPU."""
        if self.world == 1:
            return part
        return self.runner.gather_cols(part, [(N * r // self.world, N * (r + 1) // self.world) for r in range(self.world)], N)
