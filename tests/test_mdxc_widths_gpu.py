"""MDX23C (TFC_TDF_net, csrc/tfc_net.cu) at the released channel widths of MDX23C-8KFFT-InstVoc_HQ (128 -> 768 channels, 5 scales) against float64.

test_mdxc_gpu.py runs a 16/32/48-channel golden, at which the weight blocking (`umma_*_choose`: kc / n_c from Cin / Cout) and most of the
epilogue options of the tensor-core pair pipeline are never exercised.  Here:
  (a) every (operator, Cin, Cout, epilogue) the released geometry instantiates, through b200sep_selftest_umma_ex / b200sep_selftest_instnorm_act,
      against float64 PyTorch on the same device.  Gate 5e-5 of max|ref| (test_umma_gpu.py); channels outside an output slice must come back bit-exact;
  (b) the whole network at the released widths on a reduced plane (dim_f 1024, dim_t 128) against the float64 oracle, 1e-4 of max|ref| per item,
      and one item alone bit-identical to the same item inside a batch;
  (c) one full-size chunk (n_fft 8192, dim_f 4096, dim_t 256): spectrogram 1e-4 of max|ref|, audio 1e-4 max-abs (the BASELINE gate).
The create-validation test at the end needs no GPU: tfcnet_create checks its arguments before the first CUDA call."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import mdx_oracle as M
import mdxc_oracle as X

B200SEP_ERR_ARG = -1  # include/b200sep.h

# final_conv.2 gain of the full-size chunk test: make_weights(MDXCConfig(), seed=4) with synth_music(chunk, seed=8) normalised to 0.9 peaks at
# 0.2438 in the float64 oracle's audio at gain 1 (X.net_forward on the CPU); the network is linear after final_conv.2, so 0.5 / 0.2438 puts the
# separated audio's peak at 0.5 and the 1e-4 absolute audio gate means what it means for real programme material.
FULL_SIZE_OUT_GAIN = 2.05

WIDTHS = (128, 256, 384, 512, 640, 768)  # c + i*g, i = 0..5: every scale of the released network, bottleneck included
KINDS = {"conv3": 0, "pw": 1, "down": 2, "up": 3}


@pytest.fixture(scope="module")
def lib(lib_built):
    from audio_separator.separator.b200 import _lib

    return _lib


@pytest.fixture(scope="module")
def cuda(lib):
    assert torch.cuda.is_available()
    return lib


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def rel_err(got, ref):
    return (got.double() - ref.double()).abs().max().item() / max(1e-30, ref.double().abs().max().item())


def _case(kind, cin, cout, B, T, Fq, act=0, res=False, mul=False, c_total=0, c_off=0, f32=False, what=""):
    tag = f"{kind}-{cin}to{cout}-B{B}T{T}F{Fq}" + (f"-act{act}" if act else "") + ("-res" if res else "") + ("-mul" if mul else "")
    tag += (f"-ch{c_off}of{c_total}" if c_total else "") + ("-f32" if f32 else "") + (f"-{what}" if what else "")
    return pytest.param(kind, cin, cout, B, T, Fq, act, res, mul, c_total, c_off, f32, id=tag)


def _operator_cases():
    small = [(4, 32), (1, 8), (4, 8), (1, 32)]  # (T, F) planes as small as the network's deepest scales; F = 8 and 32 leave the 112 / 128 pixel tiles ragged
    cs = [_case("pw", 16, 128, 2, 2, 136, what="first_conv")]  # F 136: one full 128-row tile and a ragged one
    for i, c in enumerate(WIDTHS):
        T, Fq = small[i % 4]
        cs.append(_case("pw", c, c, 2, T, Fq, what="shortcut"))
        cs.append(_case("pw", 2 * c, c, 2, T, Fq, what="dec_shortcut"))
        cs.append(_case("conv3", c, c, 2, T, Fq, what="tfc1"))
        cs.append(_case("conv3", 2 * c, c, 2, T, Fq, what="dec_tfc1"))
        cs.append(_case("conv3", c, c, 2, *small[(i + 1) % 4], res=True, what="tfc2"))
    cs += [
        _case("pw", 144, 128, 2, 4, 32, act=2, what="final_conv0"),
        _case("pw", 128, 32, 2, 4, 136, f32=True, what="final_conv2"),
        _case("pw", 128, 128, 2, 1, 136, act=2, res=True, mul=True, c_total=144, c_off=16, what="all_options"),  # every pw option at once
        _case("conv3", 128, 128, 2, 4, 136, res=True, c_total=256, c_off=128, what="enc0_into_cat"),  # encoder output -> second half of CAT
        _case("conv3", 640, 640, 2, 1, 32, res=True, c_total=1280, c_off=640, what="enc4_into_cat"),
        _case("conv3", 128, 128, 2, 4, 136, res=True, mul=True, c_total=144, c_off=16, what="last_dec_block"),  # tfc2 + shortcut, * first_conv, into FC
        _case("conv3", 128, 128, 2, 1, 8, res=True, mul=True, c_total=144, c_off=16, what="last_dec_block"),
    ]
    for i, c in enumerate(WIDTHS[:-1]):
        cs.append(_case("down", c, c + 128, 2, 4 if i % 2 else 2, 16 if i % 2 else 136, what="downscale"))
    for i, c in enumerate(WIDTHS[1:]):
        o = c - 128
        cs.append(_case("up", c, o, 2, 1 if i % 2 else 2, 8 if i % 2 else 16, c_total=2 * o, c_off=0, what="upscale_into_cat"))
    cs.append(_case("up", 256, 128, 2, 2, 16, res=True, c_total=256, c_off=128, what="skip_mul"))
    return cs


def _reference(kind, x, w, act, res, mul):
    if kind == "conv3":
        y = F.conv2d(x, w, padding=1)
    elif kind == "pw":
        y = F.conv2d(x, w[:, :, None, None])
    elif kind == "down":
        y = F.conv2d(x, w, stride=2)
    else:
        y = F.conv_transpose2d(x, w, stride=2)
    if act == 1:
        y = torch.relu(y)
    elif act == 2:
        y = F.gelu(y)
    if res is not None:
        y = y * res if kind == "up" else y + res
    if mul is not None:
        y = y * mul
    return y


@pytest.mark.gpu
@pytest.mark.timeout(120)
@pytest.mark.parametrize("kind,cin,cout,B,T,Fq,act,res,mul,c_total,c_off,f32", _operator_cases())
def test_umma_epilogue_at_released_widths_vs_float64(cuda, kind, cin, cout, B, T, Fq, act, res, mul, c_total, c_off, f32):
    g = torch.Generator(device="cuda").manual_seed(cin * 7919 + cout * 31 + T * 5 + Fq + KINDS[kind])
    x = torch.randn(B, cin, T, Fq, device="cuda", generator=g)
    taps = {"conv3": 9, "pw": 1, "down": 4, "up": 4}[kind]
    wshape = {"conv3": (cout, cin, 3, 3), "pw": (cout, cin), "down": (cout, cin, 2, 2), "up": (cin, cout, 2, 2)}[kind]
    w = (torch.randn(*wshape, device="cuda", generator=g) / (taps * cin) ** 0.5).cpu().contiguous()
    To, Fo = {"down": (T // 2, Fq // 2), "up": (2 * T, 2 * Fq)}.get(kind, (T, Fq))
    r = torch.randn(B, cout, To, Fo, device="cuda", generator=g) if res else None
    m = torch.randn(B, cout, To, Fo, device="cuda", generator=g) if mul else None
    ct = c_total or cout
    out = torch.full((B, ct, To, Fo), 7.0, device="cuda")  # 7.0 is exact in the bf16 pair: it must survive outside the slice bit for bit
    out[:, c_off : c_off + cout] = float("nan")
    rc = cuda.lib.b200sep_selftest_umma_ex(KINDS[kind], x.data_ptr(), w.data_ptr(), r.data_ptr() if res else None, m.data_ptr() if mul else None, out.data_ptr(),
                                           B, cin, cout, T, Fq, act, c_total, c_off, int(f32), None)
    cuda.check(rc, "selftest_umma_ex")
    ref = _reference(kind, x.double(), w.cuda().double(), act, r.double() if res else None, m.double() if mul else None)
    got = out[:, c_off : c_off + cout]
    outside = torch.cat([out[:, :c_off], out[:, c_off + cout :]], 1)
    assert torch.isfinite(got).all()
    assert bool((outside == 7.0).all()), "channels outside the output slice were written"
    err = rel_err(got, ref)
    print(f"{kind} {cin}->{cout}: rel err {err:.2e}")
    assert err <= 5e-5


@pytest.mark.gpu
@pytest.mark.timeout(120)
@pytest.mark.parametrize(
    "B,Cn,c_total,c_off,P,act",
    [
        (2, 16, 16, 0, 8, 2),
        (2, 768, 768, 0, 8, 2),  # TDF hidden plane of the reduced-plane bottleneck (4 x 8 / bn)
        (2, 128, 256, 128, 4096, 2),  # down_norm: channels [c, 2c) of CAT
        (2, 640, 1280, 640, 32, 0),
        (1, 32, 48, 8, 8192, 0),
        (1, 16, 16, 0, 262144, 2),  # a full-size scale-0 plane, 256 frames x 1024 bins
        (1, 8, 24, 16, 262144, 0),
    ],
)
def test_instnorm_act_vs_float64(cuda, B, Cn, c_total, c_off, P, act):
    g = torch.Generator(device="cuda").manual_seed(B + Cn + c_total + c_off + P + act)
    x = torch.randn(B, c_total, P, device="cuda", generator=g) * 3 + torch.randn(1, c_total, 1, device="cuda", generator=g) * 4  # per-channel offsets
    gamma = torch.rand(Cn, device="cuda", generator=g) + 0.5
    beta = torch.randn(Cn, device="cuda", generator=g) * 0.3
    out = torch.full((B, Cn, P), float("nan"), device="cuda")
    rc = cuda.lib.b200sep_selftest_instnorm_act(x.data_ptr(), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(), B, Cn, c_total, c_off, P, act, None)
    cuda.check(rc, "selftest_instnorm_act")
    ref = F.instance_norm(x[:, c_off : c_off + Cn].double(), weight=gamma.double(), bias=beta.double(), eps=1e-5)
    if act == 2:
        ref = F.gelu(ref)
    assert torch.isfinite(out).all()
    err = rel_err(out, ref)
    print(f"instnorm B={B} C={Cn} P={P}: rel err {err:.2e}")
    assert err <= 5e-5


def _tfcnet(cfg, w, max_batch):
    from audio_separator.separator.b200 import engine

    return engine.TfcNet(w, cfg.dim_f, cfg.dim_t, cfg.num_subbands, 2, cfg.num_scales, cfg.num_blocks_per_scale, cfg.num_channels_model, cfg.growth,
                         cfg.bottleneck_factor, cfg.num_targets, max_batch=max_batch)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_released_widths_reduced_plane_vs_float64(cuda):
    """c = g = 128, 5 scales, 2 blocks, bn 4, 2 targets: every layer at its released Cin / Cout.  dim_f 1024, dim_t 128: Fs 256, bottleneck plane 4 x 8;
    the TDF linears take the tensor-core GEMM at scales 0-2 and the SIMT fallback at scales 3-5 (Fs >> i / bn < 16)."""
    cfg = X.MDXCConfig(dim_f=1024, dim_t=128)
    w = X.make_weights(cfg, seed=11)
    net = _tfcnet(cfg, w, max_batch=2)
    x = (np.random.default_rng(12).standard_normal((3, 4, cfg.dim_f, cfg.dim_t)) * 2).astype(np.float32)
    torch.set_num_threads(min(32, os.cpu_count() or 8))
    ref = X.net_forward_spec(w, cfg, x, dtype="float64")  # (3, S*4, dim_f, dim_t)

    def run(xb):  # three items through max_batch 2: the last sub-batch is smaller than the batch the TMA plans were bound for
        return net.forward_spec(dev(xb.transpose(0, 1, 3, 2))).cpu().numpy().transpose(0, 1, 2, 4, 3).reshape(xb.shape[0], *ref.shape[1:])

    got = run(x)
    errs = [float(np.abs(got[i].astype(np.float64) - ref[i]).max() / np.abs(ref[i]).max()) for i in range(3)]
    print("reduced-plane network, rel err per item: " + " ".join(f"{e:.2e}" for e in errs))
    assert max(errs) <= 1e-4, errs
    alone = run(x[:1])
    assert np.array_equal(alone[0], got[0]), "item 0 alone differs from item 0 inside a batch of 2"


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_full_size_chunk_vs_float64(cuda):
    from audio_separator.separator.b200 import engine

    cfg = X.MDXCConfig()
    w = X.make_weights(cfg, seed=4, out_gain=FULL_SIZE_OUT_GAIN)
    net = _tfcnet(cfg, w, max_batch=1)
    eng = engine.MdxcEngine(net, cfg.n_fft, cfg.hop_length, cfg.dim_f, cfg.dim_t, cfg.overlap)
    mix = M.normalize(M.synth_music(cfg.chunk_size, seed=8), 0.9, 0.0)
    torch.set_num_threads(min(32, os.cpu_count() or 8))
    # X.net_forward(w, cfg, mix[None], "float64"), keeping the spectrogram it passes through
    spec = M.stft_forward(mix[None], cfg.n_fft, cfg.hop_length, cfg.dim_f)  # (1, 4, dim_f, dim_t)
    ref_spec = X.net_forward_spec(w, cfg, spec, dtype="float64")
    ref_audio = M.stft_inverse(ref_spec.reshape(1, cfg.num_targets, 4, cfg.dim_f, cfg.dim_t), cfg.n_fft, cfg.hop_length)  # (1, S, 2, chunk)
    assert 0.3 < np.abs(ref_audio).max() < 1.0  # the gain brings the audio to a real signal level: 1e-4 absolute is then a meaningful gate

    got_spec = net.forward_spec(dev(spec.transpose(0, 1, 3, 2))).cpu().numpy().transpose(0, 1, 2, 4, 3).reshape(ref_spec.shape)
    es = float(np.abs(got_spec.astype(np.float64) - ref_spec).max() / np.abs(ref_spec).max())
    got_audio = eng.model_run(dev(mix[None])).cpu().numpy()
    assert got_audio.shape == ref_audio.shape == (1, cfg.num_targets, 2, cfg.chunk_size)
    ea = float(np.abs(got_audio.astype(np.float64) - ref_audio).max())
    print(f"full-size chunk: spectrogram rel err {es:.2e}, audio max-abs err {ea:.2e} (peak {np.abs(ref_audio).max():.3f})")
    assert es <= 1e-4
    assert ea <= 1e-4


def test_create_rejects_a_bottleneck_tdf_plane_the_instance_norm_cannot_take(lib):
    """The instance norm of the TDF hidden layer needs planes of a multiple of 8 elements; at the bottleneck that plane is (dim_t >> n) * ((Fs >> n) / bn).
    tfcnet_create must refuse a geometry where it is not, instead of creating a network whose every forward fails."""

    def create(dim_t):
        cfg = lib.TfcNetConfig(128, dim_t, 4, 2, 2, 2, 16, 16, 4, 2, 1)  # Fs 32, 2 scales: bottleneck F 8, TDF hidden width 8 / bn = 2
        n = lib.lib.b200sep_tfcnet_param_count(C.byref(cfg))
        blob = np.zeros(n, np.float32)
        h = C.c_void_p()
        rc = lib.lib.b200sep_tfcnet_create(C.byref(h), C.byref(cfg), blob.ctypes.data_as(C.c_void_p), n)
        msg = lib.lib.b200sep_last_error().decode(errors="replace")
        if rc == 0:
            lib.lib.b200sep_tfcnet_destroy(h)
        return rc, msg

    rc, msg = create(4)  # bottleneck T 1: plane 1 * 2
    assert rc == B200SEP_ERR_ARG and "TDF hidden plane" in msg, (rc, msg)
    rc, msg = create(16)  # bottleneck T 4: plane 4 * 2 = 8
    assert rc != B200SEP_ERR_ARG, msg
