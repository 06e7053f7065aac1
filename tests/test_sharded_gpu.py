"""GPU: the time-sharded engines (audio_separator/separator/b200/sharded.py and the `dist=` paths of MdxcEngine / DemucsEngine) through NCCL.

World size 1 (always runs on the one-GPU box): the sharded code path -- slice of the padded mixture, ShardRunner, ranged overlap-add with slice
outputs, the shared-host-buffer end-to-end entry -- must reproduce the plain engines bit for bit.  World size 2 (skipped unless two GPUs are
visible): two processes, halo exchange + gather over NVLink, compared with the single-GPU result inside rank 0."""
import os
import socket

import numpy as np
import pytest
import torch

import mdx_oracle as O

pytestmark = pytest.mark.gpu

SMALL = dict(n_fft=1536, hop_length=256, dim_f=768, dim_t=32, segment_size=32, g=8)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _mdx_pair(cfg, batch, sharded_cls, precision=1):
    from audio_separator.separator.b200 import engine, mdx_weights

    w = O.make_convtdfnet_weights(cfg, seed=3, out_gain=0.05)
    hp = mdx_weights.infer_hparams_from_state(w)
    net = engine.MdxNet(mdx_weights.flatten_state(w, **hp), dim_t=cfg.dim_t, max_batch=batch, precision=precision, **hp)
    args = (net, cfg.n_fft, cfg.hop_length, cfg.dim_f, cfg.segment_size, cfg.overlap, cfg.compensate)
    return engine.MdxEngine(*args, batch_size=batch), sharded_cls(*args, batch_size=batch)


def _demucs_small():
    from fractions import Fraction

    import demucs_oracle as D
    from audio_separator.separator.b200 import demucs as dm

    kw = dict(channels=8, bottom_channels=32, t_layers=3, t_heads=4, segment=Fraction(1, 2))
    ocfg = D.HTConfig(**kw)
    nets = [dm.HTDemucsNet(dm.HTDemucsConfig(**kw), D.make_weights(ocfg, seed=5 + i)) for i in range(2)]
    return dm, ocfg, nets


def _mdxc_small():
    import mdxc_oracle as X
    from audio_separator.separator.b200 import engine

    cfg = X.MDXCConfig(n_fft=1024, hop_length=256, dim_f=512, dim_t=16, num_scales=2, num_channels_model=16, growth=16, bottleneck_factor=4, overlap=4)  # the golden's small geometry
    w = X.make_weights(cfg, seed=4, out_gain=0.3)
    net = engine.TfcNet(w, cfg.dim_f, cfg.dim_t, cfg.num_subbands, 2, cfg.num_scales, cfg.num_blocks_per_scale, cfg.num_channels_model, cfg.growth, cfg.bottleneck_factor, cfg.num_targets, max_batch=3)
    return engine, cfg, net


def _check_all(rank, world, results):
    """Runs on every rank of an initialised nccl group; rank 0 appends (name, bit_identical, max_abs_diff)."""
    import torch.distributed as dist
    from audio_separator.separator.b200.sharded import ShardedMdxEngine

    dev = torch.device("cuda", torch.cuda.current_device())
    # ---- MDX: device-resident and shared-host-buffer entries
    cfg = O.MDXConfig(**SMALL)
    n = 9 * cfg.chunk_size // 2 + 321
    mix = torch.from_numpy(O.synth_music(n, seed=2)).to(dev)
    single, sharded = _mdx_pair(cfg, 2, ShardedMdxEngine)
    got = sharded.separate_device(mix, 0.9, 0.0)
    if world == 1:
        mh = torch.from_numpy(O.synth_music(n, seed=2)).pin_memory()
        outs = [torch.empty((n, 2)).pin_memory() for _ in range(2)]
        sharded.separate_host(mh, outs[0], outs[1], 0.9, 0.0)
    if rank == 0:
        ref = single.separate_device(mix, 0.9, 0.0)
        for name, g, r in (("mdx primary", got[0], ref[0]), ("mdx secondary", got[1], ref[1])):
            results.append((name, bool(torch.equal(g, r)), float((g - r).abs().max())))
        if world == 1:
            for name, g, r in (("mdx host primary", outs[0].to(dev), ref[0]), ("mdx host secondary", outs[1].to(dev), ref[1])):
                results.append((name, bool(torch.equal(g, r)), float((g - r).abs().max())))
    # ---- MDX23C
    engine, xcfg, net = _mdxc_small()
    n2 = 11 * xcfg.chunk_size // 2 + 77
    mix2 = torch.from_numpy(O.synth_music(n2, seed=6)).to(dev)
    es = engine.MdxcEngine(net, xcfg.n_fft, xcfg.hop_length, xcfg.dim_f, xcfg.dim_t, xcfg.overlap, dist=dist)
    got2 = es.gather(es.demix_device(mix2), n2)
    if rank == 0:
        ref2 = engine.MdxcEngine(net, xcfg.n_fft, xcfg.hop_length, xcfg.dim_f, xcfg.dim_t, xcfg.overlap).demix_device(mix2)
        results.append(("mdx23c", bool(torch.equal(got2, ref2)), float((got2 - ref2).abs().max())))
    # ---- Demucs: bag of 2, shifts 2
    dm, ocfg, nets = _demucs_small()
    n3 = 7 * ocfg.seg_len + 1234
    mix3 = torch.from_numpy(O.synth_music(n3, seed=8)).to(dev)
    offs = [[1000, 15000], [22050, 7]]
    bag = [[1.0, 0.5, 0.0, 2.0], [0.0, 0.5, 1.0, 1.0]]
    ed = dm.DemucsEngine(nets, bag_weights=bag, batch_size=3, dist=dist)
    got3 = ed.gather(ed.demix_device(mix3, offs), n3)
    if rank == 0:
        ref3 = dm.DemucsEngine(nets, bag_weights=bag, batch_size=3).demix_device(mix3, offs)
        results.append(("demucs", bool(torch.equal(got3, ref3)), float((got3 - ref3).abs().max())))
    dist.barrier()


def _worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    res = []
    _check_all(rank, world, res)
    if rank == 0:
        q.put(res)
    dist.destroy_process_group()


def _run(world):
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
    codes = [p.exitcode for p in procs]
    for p in procs:  # a rank that died leaves its peers waiting in NCCL: do not let them hold the GPUs
        if p.is_alive():
            p.kill()
    assert codes == [0] * world, codes
    return q.get(timeout=10)


@pytest.mark.timeout(900)
def test_sharded_engines_world1_equal_plain_engines(lib_built):
    for name, same, diff in _run(1):
        assert same and diff == 0.0, (name, diff)


@pytest.mark.timeout(900)
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_engines_world2_equal_single_gpu(lib_built):
    for name, same, diff in _run(2):
        # per-sample arithmetic is the single-GPU arithmetic (same contributions, same order).  The ranks batch their segments differently from the
        # single-GPU run; every reduction inside a forward is partitioned independently of the batch size (GroupNorm since round 2), so the Demucs
        # result is expected to agree to the last bits -- the gate leaves room for one reduction that is not (4e-6 was seen before that change)
        assert diff <= 1e-5, (name, diff)
        if name.startswith("mdx"):
            assert same, name
