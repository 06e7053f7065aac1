"""CPU: time-sharding of the Roformer chunk list (b200/sharded.py plan_start_shards).  The Roformer grid is not regular: chunks sit every `step`
samples and the tail is clamped to N - chunk, so with step < chunk the last start repeats.  Planner properties, and the Hamming overlap-add of the
planned shards through ShardRunner over gloo (world 2, 3) against the single-process result."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist

from test_sharding_cpu import _spawn

SR = 44100


def roformer_starts(N, C, step):  # mdxc_separator.py:310-315 (RoformerEngine.chunk_starts)
    return [i if i + C <= N else N - C for i in range(0, N, step)]


C_EP317 = 441 * 800  # hop 441, dim_t 801: 8-s chunks
GRIDS = {
    "step == chunk (overlap 8)": (3 * 60 * SR + 12345, C_EP317, min(8 * SR, C_EP317)),
    "step < chunk (overlap 3 s, repeated tail)": (100 * SR + 777, C_EP317, 3 * SR),
    "step < chunk (overlap 0.03)": (120 * SR + 5, C_EP317, int(0.03 * SR)),
    "ep_317, 5-min track": (5 * 60 * SR, C_EP317, min(8 * SR, C_EP317)),
}


def _check_plan(shards, starts, C, N, world):
    assert len(shards) == world
    assert shards[0].q0 == 0 and shards[-1].q1 == N and all(a.q1 == b.q0 for a, b in zip(shards, shards[1:]))  # [0, N) exactly once
    assert shards[0].c0 == 0 and shards[-1].c1 == len(starts) and all(a.c1 == b.c0 for a, b in zip(shards, shards[1:]))  # every unit owned once
    assert shards[0].halo == 0 and shards[-1].send == 0 and all(a.send == b.halo for a, b in zip(shards, shards[1:]))
    for s in shards:
        assert all(s.q0 <= starts[i] < s.q1 for i in range(s.c0, s.c1))  # a unit belongs to the rank its first sample falls in
        need = [i for i, st in enumerate(starts) if st < s.q1 and st + C > s.q0]
        if s.q1 > s.q0:
            assert s.c0 - s.halo == need[0] and need[-1] < s.c1  # every covering unit is local, and the halo is no larger than needed
        if s.rank > 0:
            assert s.c0 - s.halo >= shards[s.rank - 1].c0  # the halo comes from the left neighbour alone


@pytest.mark.parametrize("name", list(GRIDS))
def test_plan_start_shards_properties(name):
    from audio_separator.separator.b200.sharded import plan_start_shards

    N, C, step = GRIDS[name]
    starts = roformer_starts(N, C, step)
    if step < C:
        assert starts[-1] == starts[-2] == N - C  # the clamped tail repeats
    if name.startswith("ep_317"):
        assert len(starts) == 38 and starts[-1] == N - C and starts[-2] == 36 * C
    for world in (1, 2, 4, 8):
        _check_plan(plan_start_shards(N, world, starts, C), starts, C, N, world)


def test_plan_start_shards_too_short_and_bad_grid():
    from audio_separator.separator.b200.sharded import plan_start_shards

    C = 1000
    starts = roformer_starts(2500, C, C)  # [0, 1000, 1500]
    with pytest.raises(ValueError, match="too short"):
        plan_start_shards(2500, 8, starts, C)  # ranges of ~312 samples, chunks of 1000: a halo would span several ranks
    plan_start_shards(2500, 2, starts, C)
    with pytest.raises(ValueError):
        plan_start_shards(2500, 2, [0, 1500, 1000], C)  # not sorted
    with pytest.raises(ValueError):
        plan_start_shards(2500, 2, [], C)


def test_plan_range_shards_is_the_stride_form():
    from audio_separator.separator.b200.sharded import plan_range_shards, plan_start_shards

    for n_out, world, n_units, stride, ulen, base in ((26_460_000, 8, 818, 32640, 261120, 228480), (1000, 3, 63, 16, 64, 48), (13_230_000, 4, 52, 257985, 343980, 21273)):
        a = plan_range_shards(n_out, world, n_units, stride, ulen, base)
        assert a == plan_start_shards(n_out, world, [i * stride - base for i in range(n_units)], ulen)


def ola_starts_np(units, first, starts, window, q0, q1):
    """The gather of ola_starts_kernel restated in float32: local units[0] is global unit `first`; the covering units of every sample are added in
    ascending order, acc / max(cnt, 1e-10)."""
    C = units.shape[-1]
    acc = np.zeros((units.shape[1], q1 - q0), np.float32)
    cnt = np.zeros(q1 - q0, np.float32)
    for j in range(units.shape[0]):
        s = starts[first + j]
        a, b = max(s, q0), min(s + C, q1)
        if b > a:
            w = window[a - s : b - s]
            acc[:, a - q0 : b - q0] += units[j][:, a - s : b - s] * w
            cnt[a - q0 : b - q0] += w
    return acc / np.maximum(cnt, np.float32(1e-10))


def _roformer_worker(rank, world, port, N, C, step, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from audio_separator.separator.b200.sharded import ShardRunner, plan_start_shards

    starts = roformer_starts(N, C, step)
    units = np.random.default_rng(11).standard_normal((len(starts), 4, C)).astype(np.float32)  # 2 stems x stereo
    window = np.hamming(C).astype(np.float32)
    runner = ShardRunner(dist)
    sh = plan_start_shards(N, world, starts, C)[rank]
    local = torch.zeros((sh.halo + sh.n_own, 4, C))

    def compute(buf, slot0, unit0, n):  # stands in for the Roformer forward of the chunks [unit0, unit0 + n)
        buf[slot0 : slot0 + n] = torch.from_numpy(units[unit0 : unit0 + n])

    runner.wait_all(runner.run_units(sh, local, compute, max_batch=2))
    mine = ola_starts_np(local.numpy(), sh.c0 - sh.halo, starts, window, sh.q0, sh.q1)
    full = runner.gather_cols(torch.from_numpy(mine), [(N * r // world, N * (r + 1) // world) for r in range(world)], N)
    if rank == 0:
        ref = ola_starts_np(units, 0, starts, window, 0, N)
        q.put(float(np.abs(full.numpy() - ref).max()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world,N,C,step", [(2, 1000, 64, 64), (3, 1000, 64, 64), (2, 1003, 64, 24), (3, 1003, 64, 24), (3, 997, 90, 7)])
def test_roformer_sharded_overlap_add_is_exact(world, N, C, step):
    assert _spawn(_roformer_worker, world, N, C, step) == 0.0  # same contributions in the same order per output sample
