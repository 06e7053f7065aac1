"""GPU: the time-sharded Roformer path -- b200sep_overlap_add_starts_range and RoformerEngine(dist=) through NCCL.

Kernel: the full range against a float64 restatement, every slice of a 3-way split against the full call's columns (bit for bit), and the argument
check for outputs that need a chunk the buffer does not hold.  World size 1: the sharded engine reproduces the plain one bit for bit (BS-Roformer and
Mel-Band, 1 and 2 stems, overlap 8 and 0.03) and the MDXC plugin writes the same files with and without `b200_sharded`.  World size 2 (skipped
unless two GPUs are visible): halo exchange + gather over NVLink, compared with the single-GPU result inside rank 0."""
import os
import socket
import wave as wavmod

import numpy as np
import pytest
import torch

import mdx_oracle as M
import roformer_oracle as R

pytestmark = pytest.mark.gpu

SMALL = dict(dim=32, depth=2, time_transformer_depth=1, freq_transformer_depth=2, freqs_per_bands=(2, 2, 4, 4, 8, 12, 16, 17), dim_head=8, heads=4, stft_n_fft=128,
             stft_hop_length=32, stft_win_length=128)
MSMALL = dict(dim=32, depth=2, time_transformer_depth=1, freq_transformer_depth=1, num_bands=12, dim_head=8, heads=4, mask_estimator_depth=2, stft_n_fft=128, stft_hop_length=32,
              stft_win_length=128)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_overlap_add_starts_range_kernel(lib_built):
    from audio_separator.separator.b200._lib import check, lib

    g = torch.Generator().manual_seed(4)
    C, N, step, ch = 50, 233, 17, 3
    starts = [i if i + C <= N else N - C for i in range(0, N, step)]  # step < chunk: the clamped tail start repeats
    assert starts.count(N - C) >= 3
    n = len(starts)
    chunks = torch.randn((n, ch, C), generator=g)
    win = torch.from_numpy(np.hamming(C).astype(np.float32))
    cd, wd, sd = chunks.cuda(), win.cuda(), torch.tensor(starts, dtype=torch.int64).cuda()
    full = torch.empty((ch, N), device="cuda")
    check(lib.b200sep_overlap_add_starts_range(cd.data_ptr(), sd.data_ptr(), wd.data_ptr(), 0, n, n, ch, C, N, 0, N, full.data_ptr(), N, 0, 0), "overlap_add_starts_range")
    res, cnt = torch.zeros((ch, N), dtype=torch.float64), torch.zeros(N, dtype=torch.float64)
    for i, s in enumerate(starts):
        res[:, s : s + C] += chunks[i].double() * win.double()
        cnt[s : s + C] += win.double()
    assert (full.cpu().double() - res / cnt.clamp(min=1e-10)).abs().max() <= 1e-6
    old = torch.empty((ch, N), device="cuda")  # the whole-track entry is the full-range call
    check(lib.b200sep_overlap_add_starts(cd.data_ptr(), sd.data_ptr(), wd.data_ptr(), n, ch, C, N, old.data_ptr(), 0), "overlap_add_starts")
    assert torch.equal(old, full)
    # 3-way split: each rank's chunks [c0 - halo, c1) and its output slice with its own leading dimension
    from audio_separator.separator.b200.sharded import plan_start_shards

    for sh in plan_start_shards(N, 3, starts, C):
        first, n_local, n_q = sh.c0 - sh.halo, sh.halo + sh.n_own, sh.q1 - sh.q0
        loc = cd[first : first + n_local].contiguous()
        part = torch.full((ch, n_q + 5), float("nan"), device="cuda")  # leading dimension n_q + 5; the 5 padding columns stay untouched
        check(lib.b200sep_overlap_add_starts_range(loc.data_ptr(), sd.data_ptr(), wd.data_ptr(), first, n_local, n, ch, C, N, sh.q0, sh.q1, part.data_ptr(), n_q + 5, sh.q0, 0),
              "overlap_add_starts_range")
        assert torch.equal(part[:, :n_q], full[:, sh.q0 : sh.q1]) and bool(part[:, n_q:].isnan().all())
        if sh.rank == 2:  # the last rank holds the repeated tail starts
            assert starts[sh.c1 - 1] == starts[sh.c1 - 2] == N - C
    # outputs that need a chunk the buffer does not hold: an error code, no read
    sh = plan_start_shards(N, 3, starts, C)[1]
    for first, n_local in ((sh.c0, sh.n_own), (sh.c0 - sh.halo, sh.halo + sh.n_own - 1)):
        loc = cd[first : first + n_local].contiguous()
        out = torch.empty((ch, sh.q1 - sh.q0), device="cuda")
        rc = lib.b200sep_overlap_add_starts_range(loc.data_ptr(), sd.data_ptr(), wd.data_ptr(), first, n_local, n, ch, C, N, sh.q0, sh.q1, out.data_ptr(), sh.q1 - sh.q0, sh.q0, 0)
        assert rc != 0 and b"outside the buffer" in lib.b200sep_last_error()
    assert lib.b200sep_overlap_add_starts_range(cd.data_ptr(), sd.data_ptr(), wd.data_ptr(), 1, n, n, ch, C, N, 0, N, full.data_ptr(), N, 0, 0) != 0  # run past the list
    torch.cuda.synchronize()


def _nets():
    from audio_separator.separator.b200 import roformer as rf

    out = []
    for stems in (1, 2):
        kw = dict(SMALL, num_stems=stems)
        out.append((f"bs {stems}-stem", rf.BSRoformerNet(rf.BSRoformerConfig(**kw), R.make_weights(R.BSRoformerConfig(**dict(kw, dim_t=65)), seed=3 + stems))))
        kw = dict(MSMALL, num_stems=stems)
        out.append((f"mel {stems}-stem", rf.BSRoformerNet(rf.MelBandRoformerConfig(**kw), R.make_mel_weights(R.MelBandRoformerConfig(**dict(kw, dim_t=65)), seed=6 + stems))))
    return out


def _check_engines(rank, world, results):
    """Every rank of an initialised nccl group; rank 0 appends (name, bit_identical, max_abs_diff)."""
    import torch.distributed as dist
    from audio_separator.separator.b200 import roformer as rf

    dev = torch.device("cuda", torch.cuda.current_device())
    n = 23 * 2048 + 777  # chunk 2048 (hop 32, dim_t 65)
    mix = torch.from_numpy(M.synth_music(n, seed=21)).to(dev)
    for name, net in _nets():
        for overlap in (8, 0.03):
            # batches of at most 2: balanced_batches then splits the chunk list as the plain engine does, so world 1 runs the same forwards
            es = rf.RoformerEngine(net, 65, overlap, 44100, n_instruments=2, batch_size=2, dist=dist)
            got = es.gather(es.demix_device(mix), n)
            if rank == 0:
                ref = rf.RoformerEngine(net, 65, overlap, 44100, n_instruments=2, batch_size=2).demix_device(mix)
                results.append((f"{name} overlap {overlap}", bool(torch.equal(got, ref)), float((got - ref).abs().max())))
    with pytest.raises(NotImplementedError):
        es.demix_device(mix[:, :1000])
    dist.barrier()


def _plugin_files(tmp, sharded):
    import yaml

    from audio_separator.separator import Separator

    ocfg = R.BSRoformerConfig(**dict(SMALL, dim_t=65, overlap=8))
    np.savez(os.path.join(tmp, "tiny_bs_roformer.npz"), **R.make_weights(ocfg, seed=12))
    model = dict(SMALL, freqs_per_bands=list(SMALL["freqs_per_bands"]), stereo=True, num_stems=1, mask_estimator_depth=2)
    with open(os.path.join(tmp, "tiny_bs_roformer.yaml"), "w") as f:
        yaml.safe_dump({"audio": {"sample_rate": 44100, "hop_length": 32, "n_fft": 128, "dim_f": 65}, "model": model,
                        "training": {"instruments": ["Vocals", "Instrumental"], "target_instrument": "Vocals"}, "inference": {"dim_t": 65}}, f)
    pcm = (M.synth_music(30000, seed=13).T * 32767).astype("<i2")
    with wavmod.open(os.path.join(tmp, "song.wav"), "wb") as wf:
        wf.setnchannels(2); wf.setsampwidth(2); wf.setframerate(44100); wf.writeframes(pcm.tobytes())
    out_dir = os.path.join(tmp, "out_sharded" if sharded else "out")
    params = {"batch_size": 2, "segment_size": 65, **({"b200_sharded": True} if sharded else {})}
    sep = Separator(model_file_dir=tmp, output_dir=out_dir, mdxc_params=params)
    sep.load_model("tiny_bs_roformer.npz")
    files = sep.separate(os.path.join(tmp, "song.wav"))
    return files, {f: open(os.path.join(out_dir, f), "rb").read() for f in files}


def _worker(rank, world, port, tmp, q):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    res = []
    _check_engines(rank, world, res)
    if world == 1:
        plain, sharded = _plugin_files(tmp, False), _plugin_files(tmp, True)
        res.append(("plugin files", plain[0] == sharded[0] and len(plain[0]) == 2 and plain[1] == sharded[1], 0.0))
    if rank == 0:
        q.put(res)
    dist.destroy_process_group()


def _run(world, tmp):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, str(tmp), q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
    codes = [p.exitcode for p in procs]
    for p in procs:  # a rank that died leaves its peers waiting in NCCL: do not let them hold the GPUs
        if p.is_alive():
            p.kill()
    assert codes == [0] * world, codes
    return q.get(timeout=10)


@pytest.mark.timeout(900)
def test_sharded_roformer_world1_equals_plain_engine(lib_built, tmp_path):
    res = _run(1, tmp_path)
    assert len(res) == 9
    for name, same, diff in res:
        assert same and diff == 0.0, (name, diff)


@pytest.mark.timeout(900)
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_roformer_world2_matches_single_gpu(lib_built, tmp_path):
    res = _run(2, tmp_path)
    for name, same, diff in res:
        # per-sample overlap-add arithmetic is the single-GPU arithmetic; the ranks batch their chunks differently from the single-GPU run, and a GEMM
        # may pick another kernel for another batch size, so the forwards agree to rounding, not necessarily to the bit
        print(f"{name}: bit_identical={same} max_abs={diff:.3e}")
        assert diff <= 1e-5, (name, diff)
