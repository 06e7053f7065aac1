"""Time-sharding of ONE track across the GPUs of a box (BASELINE north_star: "chunks shard by time across the 8 GPUs
with overlap-region halo exchange via NCCL").

The reference has no multi-GPU path (SURVEY.md section 2.1); this is new.  The chunked architectures all have the same
structure (SURVEY.md section 8e): independent units (MDX chunks, mdx_separator.py:335-348; MDX23C and Roformer chunks, mdxc_separator.py:310-402;
Demucs segments, demucs/apply.py:215-250) placed every `stride` samples, coupled only by the overlap-add.  Three planners:

* `plan_shards`        -- MDX: contiguous chunk ranges, rank r finalises the padded positions [c0*step, c1*step).
* `plan_range_shards`  -- MDX23C / Demucs: rank r finalises a fixed range [q0, q1) of OUTPUT samples (the same for every pass of a
                          Demucs bag / shift loop, so the accumulation order per sample is the single-GPU order and the result is
                          bit-identical); a unit belongs to the rank its first output sample falls in.
* `plan_start_shards`  -- Roformer: the same over an explicit, non-decreasing start list (the tail chunk clamped to N - chunk);
                          `plan_range_shards` is its stride form.
In each, a rank needs the trailing units of its LEFT neighbour that reach into its range: one `isend`/`irecv` pair between
time-neighbours (NCCL p2p over NVLink), posted as soon as those units are computed so the transfer overlaps the remaining forwards.
The finalised slices go to rank 0 with point-to-point receives straight into the full-size stem buffers, or -- end-to-end entry points --
every rank copies its own slice into a host buffer shared between the ranks (8 PCIe links in parallel, no gather at all).

The planners and `ShardRunner` (the control flow: unit order, halo exchange, overlap-add, gather) are pure host logic over
torch.distributed and run unchanged on CPU tensors with gloo (tests/test_sharding_cpu.py injects the compute); the engines below them
need CUDA + NCCL.
"""
from __future__ import annotations

from dataclasses import dataclass

import torch


@dataclass
class Shard:
    rank: int
    c0: int  # first own unit (chunk / segment)
    c1: int  # one past the last own unit
    halo: int  # units received from the left neighbour: [c0 - halo, c0)
    q0: int  # first output sample (unpadded coordinates) this rank finalises
    q1: int  # one past the last
    send: int = 0  # own trailing units the right neighbour needs: [c1 - send, c1)

    @property
    def n_own(self):
        return self.c1 - self.c0


def plan_shards(n_samples: int, total_len: int, step: int, chunk: int, trim: int, n_chunks: int, world: int) -> list[Shard]:
    """MDX.  Contiguous, balanced chunk ranges; rank r finalises the padded positions [c0*step, c1*step) (last rank: to the end)."""
    k = -(-chunk // step) - 1  # chunks of the left neighbour that reach into a rank's range
    base, rem = divmod(n_chunks, world)
    shards, c0 = [], 0
    for r in range(world):
        c1 = c0 + base + (1 if r < rem else 0)
        p0 = c0 * step
        p1 = total_len if r == world - 1 else c1 * step
        q0 = min(max(p0 - trim, 0), n_samples)
        q1 = min(max(p1 - trim, 0), n_samples)
        halo = min(k, c0) if c1 > c0 else 0
        shards.append(Shard(r, c0, c1, halo, q0, q1))
        c0 = c1
    for s in shards[1:]:
        left = shards[s.rank - 1]
        if s.halo > left.c1 - left.c0 and s.c1 > s.c0:
            raise ValueError(f"track too short to shard over {world} ranks: rank {s.rank} needs {s.halo} halo chunks, its neighbour owns {left.c1 - left.c0}")
        left.send = s.halo
    return shards


def plan_range_shards(n_out: int, world: int, n_units: int, stride: int, unit_len: int, base: int) -> list[Shard]:
    """MDX23C / Demucs.  Unit i covers the output samples [i*stride - base, i*stride - base + unit_len).  Rank r finalises the output samples
    [n_out*r/world, n_out*(r+1)/world) and owns the units whose first output sample (clamped into [0, n_out)) lies in that range."""
    if n_units < 1 or stride < 1 or unit_len < 1:
        raise ValueError("plan_range_shards: bad grid")
    return plan_start_shards(n_out, world, [i * stride - base for i in range(n_units)], unit_len)


def plan_start_shards(n_out: int, world: int, starts, unit_len: int) -> list[Shard]:
    """plan_range_shards over an explicit, non-decreasing start list (Roformer: the tail chunk is clamped to N - chunk, and with step < chunk several
    entries repeat it): unit i covers the output samples [starts[i], starts[i] + unit_len)."""
    from bisect import bisect_left, bisect_right

    starts = [int(s) for s in starts]
    n_units = len(starts)
    if n_units < 1 or unit_len < 1 or any(b < a for a, b in zip(starts, starts[1:])):
        raise ValueError("plan_start_shards: bad grid")
    qs = [n_out * r // world for r in range(world + 1)]
    u0 = [0] + [bisect_left(starts, qs[r]) for r in range(1, world)] + [n_units]
    shards = []
    for r in range(world):
        need_lo = 0 if r == 0 else bisect_right(starts, qs[r] - unit_len)  # first unit that reaches into [qs[r], ...)
        c0, c1 = u0[r], u0[r + 1]
        halo = max(0, c0 - need_lo) if qs[r + 1] > qs[r] else 0
        if r > 0 and halo > 0 and c0 - halo < u0[r - 1]:
            raise ValueError(f"track too short to shard over {world} ranks: rank {r} needs units from {c0 - halo}, its left neighbour owns [{u0[r - 1]}, {c0})")
        shards.append(Shard(r, c0, c1, halo, qs[r], qs[r + 1]))
    for s in shards[1:]:
        shards[s.rank - 1].send = s.halo
    return shards


def balanced_batches(n: int, max_batch: int) -> list[int]:
    """n units as ceil(n / max_batch) batches of nearly equal size (9 at max 4 -> 3+3+3, not 4+4+1: a 1-unit forward costs almost as much as a full one)."""
    if n <= 0:
        return []
    k = -(-n // max_batch)
    return [n // k + (1 if i < n % k else 0) for i in range(k)]


class ShardRunner:
    """The control flow shared by the sharded engines, over torch.distributed (nccl on the GPUs, gloo in the CPU tests).

    compute(local, slot0, unit0, n): fill local[slot0 : slot0 + n] with the outputs of the global units [unit0, unit0 + n).
    """

    def __init__(self, dist, group=None):
        self.dist, self.group = dist, group
        self.rank = dist.get_rank(group) if dist is not None else 0
        self.world = dist.get_world_size(group) if dist is not None else 1

    def _peer(self, r):
        return r if self.group is None else self.dist.get_global_rank(self.group, r)

    def run_units(self, sh: Shard, local: torch.Tensor, compute, max_batch: int):
        """Own units into local[halo:] in balanced batches; the batches holding the trailing `send` units run FIRST and the p2p pair is posted
        right after them, so the transfer to the right neighbour overlaps the remaining forwards.  Returns the outstanding requests
        (wait_all before the overlap-add)."""
        n_own = sh.n_own
        assert local.shape[0] == sh.halo + n_own
        spans, u = [], sh.c0
        for b in balanced_batches(n_own, max_batch):
            spans.append((u, b))
            u += b
        send = min(sh.send, n_own) if self.rank + 1 < self.world else 0
        head = [sp for sp in spans if sp[0] + sp[1] > sh.c1 - send] if send else []
        rest = [sp for sp in spans if sp not in head]
        reqs, posted = [], False
        for unit0, n in head:
            compute(local, sh.halo + unit0 - sh.c0, unit0, n)
        if head or sh.halo:
            reqs += self._post(sh, local)
            posted = True
        for unit0, n in rest:
            compute(local, sh.halo + unit0 - sh.c0, unit0, n)
        assert posted or (sh.halo == 0 and send == 0)
        return reqs

    def _post(self, sh: Shard, local: torch.Tensor):
        dist = self.dist
        if dist is None or self.world == 1:
            return []
        ops = []
        n = local.shape[0]
        if sh.send > 0 and self.rank + 1 < self.world:
            ops.append(dist.P2POp(dist.isend, local[n - sh.send : n], self._peer(self.rank + 1), self.group))
        if sh.halo > 0:
            ops.append(dist.P2POp(dist.irecv, local[: sh.halo], self._peer(self.rank - 1), self.group))
        return list(dist.batch_isend_irecv(ops)) if ops else []

    @staticmethod
    def wait_all(reqs):
        for r in reqs:
            r.wait()

    def gather_rows(self, bufs, shards, dim=0):
        """Rank 0 receives every other rank's finalised slice [q0, q1) along `dim` straight into its full-size buffers."""
        dist = self.dist
        if dist is None or self.world == 1:
            return
        ops = []
        me = shards[self.rank]
        if self.rank == 0:
            for s in shards[1:]:
                if s.q1 > s.q0:
                    for buf in bufs:
                        ops.append(dist.P2POp(dist.irecv, buf.narrow(dim, s.q0, s.q1 - s.q0), self._peer(s.rank), self.group))
        elif me.q1 > me.q0:
            for buf in bufs:
                ops.append(dist.P2POp(dist.isend, buf.narrow(dim, me.q0, me.q1 - me.q0), self._peer(0), self.group))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()


    def gather_cols(self, part: torch.Tensor, ranges, n_total: int):
        """part (..., q1 - q0) on every rank -> the full (..., n_total) tensor on rank 0 (None elsewhere).  Slices along the LAST axis are not
        contiguous in the destination, so rank 0 receives into per-rank staging tensors and copies them in place."""
        dist = self.dist
        part = part.contiguous()
        if self.rank != 0:
            if part.numel():
                dist.batch_isend_irecv([dist.P2POp(dist.isend, part, self._peer(0), self.group)])[0].wait()
            return None
        full = torch.empty(part.shape[:-1] + (n_total,), dtype=part.dtype, device=part.device)
        full[..., ranges[0][0] : ranges[0][1]] = part
        stage, ops = [], []
        for r in range(1, self.world):
            q0, q1 = ranges[r]
            if q1 > q0:
                t = torch.empty(part.shape[:-1] + (q1 - q0,), dtype=part.dtype, device=part.device)
                stage.append((q0, q1, t))
                ops.append(dist.P2POp(dist.irecv, t, self._peer(r), self.group))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        for q0, q1, t in stage:
            full[..., q0:q1] = t
        return full


# =========================================================================================================== MDX
from .engine import MdxEngine, _ptr, _stream, check, lib  # noqa: E402  (the planners above stay importable on their own)


class ShardedMdxEngine(MdxEngine):
    """MdxEngine whose demix runs on torch.distributed ranks (backend nccl, one process per GPU).  Every rank is given the same (2, N) mix
    (`separate_device`), or reads only its part of a host buffer shared between the ranks (`separate_host`); stems are returned on rank 0."""

    def __init__(self, *args, group=None, **kw):
        super().__init__(*args, **kw)
        import torch.distributed as dist

        if not dist.is_initialized():
            raise RuntimeError("ShardedMdxEngine needs torch.distributed to be initialised (backend nccl)")
        self.runner = ShardRunner(dist, group)
        self.dist, self.group, self.rank, self.world = dist, group, self.runner.rank, self.runner.world

    def _plan(self, N, is_match_mix=False):
        L, step, n_chunks, overlap = self.grid(N, is_match_mix)
        shards = plan_shards(N, L, step, self.chunk_size, self.trim, n_chunks, self.world)
        sh = shards[self.rank]
        p0 = sh.c0 * step  # padded positions [p0, p1) = what this rank's chunks read
        p1 = min(L, (sh.c1 - 1) * step + self.chunk_size) if sh.n_own else p0
        return L, step, n_chunks, overlap, shards, sh, p0, p1

    def _chunks_and_ola(self, sl, p0, N, is_match_mix, out_scale, primary, secondary, out_base, mix, mix_ld, mix_base):
        """Own chunks from `sl` = the padded mixture's positions [p0, p0 + len), halo exchange, overlap-add of this rank's output range [q0, q1)
        into primary / secondary rows [q - out_base]."""
        L, step, n_chunks, overlap, shards, sh, _, _ = self._plan(N, is_match_mix)
        T = self.chunk_size
        local = torch.empty((sh.halo + sh.n_own, 2, T), dtype=torch.float32, device=self.device)  # [halo | own]
        net = None if is_match_mix else self.net.handle
        Ls = sl.shape[1]

        def compute(buf, slot0, unit0, n):
            work = self._workspace(n)
            off = unit0 * step - p0
            check(lib.b200sep_mdx_run_model(self.plan.handle, net, sl.data_ptr() + off * 4, step, Ls, Ls - off, n, T, self.dim_f, int(self.enable_denoise),
                                            _ptr(buf[slot0 : slot0 + n]), _ptr(work), _stream()), "mdx_run_model")

        self.runner.wait_all(self.runner.run_units(sh, local, compute, self.batch))
        if sh.q1 > sh.q0:
            check(lib.b200sep_demix_overlap_add_range_ex(_ptr(local), sh.c0 - sh.halo, sh.halo + sh.n_own, n_chunks, T, step, L, self.trim, N, sh.q0, sh.q1, int(overlap != 0),
                                                         float(out_scale), _ptr(mix) if mix is not None else None, mix_ld, mix_base, self.compensate, 1, _ptr(primary),
                                                         _ptr(secondary) if secondary is not None else None, out_base, _stream()), "demix_overlap_add_range_ex")
        return shards

    def demix_device(self, mix_dev, is_match_mix=False, out_scale=1.0, with_secondary=False, interleave=True):
        assert interleave, "the sharded path produces (N, 2) stems"
        mix_dev = mix_dev.contiguous()
        N = mix_dev.shape[1]
        _, _, _, _, _, sh, p0, p1 = self._plan(N, is_match_mix)
        sl = torch.zeros((2, max(p1 - p0, 1)), dtype=torch.float32, device=self.device)  # this rank's part of [0]*trim + mix + [0]*pad (:329)
        a, b = max(p0, self.trim), min(p1, self.trim + N)
        if b > a:
            sl[:, a - p0 : b - p0] = mix_dev[:, a - self.trim : b - self.trim]
        primary = torch.empty((N, 2), dtype=torch.float32, device=self.device)
        secondary = torch.empty((N, 2), dtype=torch.float32, device=self.device) if with_secondary else None
        shards = self._chunks_and_ola(sl, p0, N, is_match_mix, out_scale, primary, secondary, 0, mix_dev if with_secondary else None, N, 0)
        self.runner.gather_rows([primary] + ([secondary] if with_secondary else []), shards, dim=0)
        if self.rank != 0:
            return (None, None) if with_secondary else None
        return (primary, secondary) if with_secondary else primary

    def separate_host(self, mix_host: torch.Tensor, out_primary: torch.Tensor, out_secondary: torch.Tensor, normalization_threshold=0.9, amplification_threshold=0.0):
        """End-to-end entry point over host buffers SHARED by the ranks (pinned): mix_host (2, N) float32; out_* (N, 2) float32.  Every rank uploads only
        the samples its chunks and its output range touch, the peak (mdx_separator.py:155) is an all-reduce(MAX) of the per-rank partial peaks, and every
        rank writes its own slice of both stems into the shared output buffers: N PCIe links in parallel, no gather.  Returns this rank's (h2d, d2h) bytes."""
        dist = self.dist
        N = mix_host.shape[1]
        _, _, _, _, _, sh, p0, p1 = self._plan(N)
        a, b = max(p0, self.trim), min(p1, self.trim + N)  # padded positions of this rank's chunks that hold real samples
        lo, hi = sh.q0, sh.q1
        if b > a:
            lo, hi = min(lo, a - self.trim), max(hi, b - self.trim)
        n_part, n_q = max(hi - lo, 0), sh.q1 - sh.q0
        part = torch.zeros((2, max(n_part, 1)), dtype=torch.float32, device=self.device)
        for c in range(2 if n_part else 0):  # contiguous row slices: true async copies out of the pinned buffer
            part[c, :n_part].copy_(mix_host[c, lo:hi], non_blocking=True)
        peak = torch.zeros(1, dtype=torch.float32, device=self.device)
        if n_q > 0:  # peak over the DISJOINT partition [q0, q1)
            own = part[:, sh.q0 - lo : sh.q1 - lo].contiguous()
            check(lib.b200sep_absmax(_ptr(own), own.numel(), _ptr(peak), _stream()), "absmax")
        dist.all_reduce(peak, op=dist.ReduceOp.MAX, group=self.group)
        min_peak = -1.0 if amplification_threshold is None else float(amplification_threshold)
        partn = torch.empty_like(part)
        check(lib.b200sep_normalize(_ptr(part), part.numel(), _ptr(peak), float(normalization_threshold), min_peak, _ptr(partn), _stream()), "normalize")
        peak_h = float(peak.item())  # `source = demix(mix) * peak` (:159): out_scale is a host float in the C ABI
        sl = torch.zeros((2, max(p1 - p0, 1)), dtype=torch.float32, device=self.device)
        if b > a:
            sl[:, a - p0 : b - p0] = partn[:, a - self.trim - lo : b - self.trim - lo]
        prim = torch.empty((max(n_q, 1), 2), dtype=torch.float32, device=self.device)
        sec = torch.empty((max(n_q, 1), 2), dtype=torch.float32, device=self.device)
        self._chunks_and_ola(sl, p0, N, False, peak_h, prim, sec, sh.q0, partn, partn.shape[1], lo)
        if n_q > 0:
            out_primary[sh.q0 : sh.q1].copy_(prim[:n_q], non_blocking=True)
            out_secondary[sh.q0 : sh.q1].copy_(sec[:n_q], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return int(2 * n_part * 4), int(2 * n_q * 2 * 4)
