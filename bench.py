"""bench.py -- real-time factor of the stem-separation hot path (BASELINE.json metric) on N B200s, or the CPU reference arm.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload mdx|htdemucs_ft|mdx23c|vr] [--also htdemucs_ft|none] [--dump-outputs DIR]

Workloads (BASELINE.json configs; there are no model files offline, so every network runs seeded synthetic weights of the released
geometry -- data: "synthetic"):
  mdx          configs[1]: UVR-MDX-NET-Inst_HQ_3 topology, 5-min stereo track, segment_size=256, overlap=0.25 -> 68 chunks.  THE DEFAULT LINE.
  htdemucs_ft  configs[2]: bag of 4 HTDemucs, 5-min track, shifts=2, overlap=0.25 -> 416 segment forwards.  Also measured by the default run
               and reported under "also" in the same JSON line (BASELINE.json's metric names both models).
  mdx23c       configs[3]: MDX23C TFC_TDF_net, 10-min track, overlap 8 -> 818 chunks (on request; 8-GPU config).
  vr           configs[4]: 9_HP2-UVR geometry, 32 x 3-min tracks, round-robin over the ranks (on request; 8-GPU config).

One step = separate the whole workload.
  value : audio-seconds / device-seconds with the input resident in HBM (CUDA events on the launch stream, max over ranks)
  e2e   : the same through the plugin-level entry point with HOST buffers: pinned input uploaded and stems downloaded inside the timed region
  parity: N > 1 -- the sharded result against a single-GPU run of the same engine on rank 0 (bit-identical expected);
          N = 1 -- the tensor-core path against the fp32 SIMT path of the same library on a 10-s excerpt (gate 1e-4).
N > 1  : one process per GPU (torchrun); chunks / segments of the ONE track are time-sharded with an overlap-region halo exchange over NCCL
         (strong scaling), audio_separator/separator/b200/sharded.py; the VR batch distributes whole tracks (no collective).
--impl reference: the reference's algorithm on the host CPU (torch-CPU restatement in oracle/; the reference package itself cannot be installed
         offline: no onnxruntime / librosa wheels), a bounded sample of the SAME chunk grid per step.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "python-audio-separator_b200"))

SR = 44100
MDX_OUT_GAIN = 66.97557067871094  # tests/golden/mdx_full_chunk.npz: the seeded full-size net then separates at a 0.5 peak, so the 1e-4 parity gates bite
METRIC = "real-time factor (audio-sec/wall-sec) @44.1kHz stereo"
DTYPE = "f32 (bf16x3-split tensor-core contractions, fp32 accumulate)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)), "source": "measured (MEASURED_PEAKS.json, sustained bf16 / copy)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def ncu_traffic(kernel_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, parsed from the committed `ncu --set full` capture of the
    same launch shape (profiles/ncu_dram_bytes.json: {key: {"bytes": ..., "source": file}}); None when no capture of this build is committed."""
    p = os.path.join(ROOT, "profiles", "ncu_dram_bytes.json")
    try:
        with open(p) as f:
            e = json.load(f).get(kernel_key)
        return (float(e["bytes"]), e.get("source")) if e else (None, None)
    except Exception:
        return None, None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx[0] if mx else None, "reasons": sorted(reasons), "samples": len(self.rows)}


class Ctx:
    """Process / device context of one rank."""

    def __init__(self, args):
        import torch

        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
        torch.cuda.set_device(self.local)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist
        assert self.world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torch.distributed.run --nproc-per-node {args.gpus}"

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, *vals):
        if self.dist is None:
            return [float(v) for v in vals]
        t = self.torch.tensor(list(vals), device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def sum_over_ranks(self, *vals):
        if self.dist is None:
            return [int(v) for v in vals]
        t = self.torch.tensor(list(vals), device="cuda", dtype=self.torch.int64)
        self.dist.all_reduce(t)
        return [int(v) for v in t]

    def shared_host(self, name, shape):
        """A float32 host buffer mapped by every rank (a /dev/shm file), page-locked in this process: N PCIe links fill / drain ONE array."""
        import numpy as np

        torch = self.torch
        n = 1
        for s in shape:
            n *= int(s)
        path = os.path.join("/dev/shm", f"b200sep_bench_{os.environ.get('MASTER_PORT', '0')}_{name}")
        if self.rank == 0:
            with open(path, "wb") as f:
                f.truncate(n * 4)
        self.barrier()
        arr = np.memmap(path, dtype=np.float32, mode="r+", shape=tuple(shape))
        t = torch.from_numpy(arr)
        # The mapping stays alive (and registered) until the process exits: a workload's buffers that were unmapped while still page-locked leave a stale
        # registration behind, and the next workload's mmap of the same size lands on the same addresses -> cudaHostRegister fails (seen at N = 2: the second
        # workload of the default run died here).
        self._shared = getattr(self, "_shared", [])
        self._shared.append((arr, t))
        rc = torch.cuda.cudart().cudaHostRegister(t.data_ptr(), n * 4, 0)
        assert int(rc) == 0, f"cudaHostRegister failed ({rc})"
        self.barrier()
        if self.rank == 0:
            os.unlink(path)  # the mappings keep it alive
        return t

    def timed(self, fn, steps, warmup):
        """`warmup` untimed + exactly `steps` timed calls, barrier + synchronize on both sides, CUDA events, max over ranks
        -> (ms per step, what the last timed call returned)."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        for _ in range(steps - 1):
            fn()  # the result is dropped before the next call, so its memory is reused as in every other step
        last = fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1))[0] / steps, last


def music(n, seed):
    """Deterministic programme material (oracle generator), a 30-s pattern tiled: far larger than L2, cheap to synthesise."""
    import numpy as np

    import mdx_oracle as O

    base = O.synth_music(min(n, 30 * SR), seed=seed)
    return np.tile(base, (1, -(-n // base.shape[1])))[:, :n].copy()


DUMP_BYTES = 60_000_000  # all the files of one --dump-outputs run stay under 64 MB


def dump_outputs(out_dir, prefix, arrays, budget):
    """Write the stems of one timed step as out_dir/<prefix>_<name>.npy (float32) for output-for-output comparison of two builds.

    `arrays`: {name: CUDA float32 tensor with time on the last axis, the same length for all}.  When they do not fit `budget` bytes, every array keeps
    the same fixed, seeded sample of time positions (sorted); the positions are written as out_dir/<prefix>_sample_index.npy (float64, exact)."""
    import numpy as np
    import torch

    if not arrays:  # a VR rank without tracks
        return
    lengths = {t.shape[-1] for t in arrays.values()}
    assert len(lengths) == 1, f"{prefix}: outputs of different lengths {sorted(lengths)}"
    n = lengths.pop()
    rows = sum(t.numel() // n for t in arrays.values())
    k = min(n, budget // (4 * rows + 8))
    idx = np.sort(np.random.default_rng(0).choice(n, k, replace=False)) if k < n else np.arange(n)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{prefix}_sample_index.npy"), idx.astype(np.float64))
    idx_d = torch.from_numpy(idx).to(next(iter(arrays.values())).device)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{prefix}_{name}.npy"), t.index_select(-1, idx_d).float().cpu().numpy())


# ======================================================================================================== MDX (the headline)
class MdxWorkload:
    name = "mdx"

    def __init__(self, args):
        self.args = args
        self.minutes = args.minutes or 5.0
        self.N = int(self.minutes * 60 * SR)
        self.audio_seconds = self.N / SR

    def config(self):
        a = self.args
        return {"workload": f"UVR-MDX-NET-Inst_HQ_3 topology (ConvTDFNet g=48, dim_f=3072, n_fft=6144), {self.minutes:g}-min 44.1 kHz stereo synthetic, segment_size=256, overlap=0.25, 68 chunks/step"
                if self.minutes == 5.0 else f"UVR-MDX-NET-Inst_HQ_3 topology, {self.minutes:g}-min 44.1 kHz stereo synthetic, segment_size=256, overlap=0.25",
                "batch": a.batch, "precision": a.precision, "l2": f"inputs larger than L2 (106 MB track, {0.15 * a.batch:.1f}-{1.2 * a.batch:.1f} GB activations per forward)",
                "parallelism": f"time-sharded chunks x{a.gpus}" if a.gpus > 1 else "single GPU"}

    def setup(self, ctx):
        import numpy as np

        import mdx_oracle as O
        from audio_separator.separator.architectures.mdx_separator import MDXSeparator

        torch = ctx.torch
        self.ctx, self.O = ctx, O
        a = self.args
        self.cfg = cfg = O.MDXConfig()
        self.w = O.make_convtdfnet_weights(cfg, seed=11, out_gain=MDX_OUT_GAIN)
        # the plugin is built exactly as Separator.load_model builds it (separator.py:867-914): a model file + model_data + arch_config
        self.tmp = tempfile.mkdtemp(prefix=f"b200sep_bench_r{ctx.rank}_")
        path = os.path.join(self.tmp, "UVR-MDX-NET-Inst_HQ_3.npz")
        np.savez(path, **self.w)
        import logging

        common = {"logger": logging.getLogger("bench"), "log_level": logging.WARNING, "torch_device": torch.device("cuda", ctx.local), "torch_device_cpu": torch.device("cpu"),
                  "torch_device_mps": None, "onnx_execution_provider": None, "model_name": "UVR-MDX-NET-Inst_HQ_3", "model_path": path,
                  "model_data": {"compensate": cfg.compensate, "mdx_dim_f_set": cfg.dim_f, "mdx_dim_t_set": 8, "mdx_n_fft_scale_set": cfg.n_fft, "primary_stem": "Instrumental"},
                  "output_format": "WAV", "output_bitrate": None, "output_dir": self.tmp, "normalization_threshold": 0.9, "amplification_threshold": 0.0,
                  "output_single_stem": None, "invert_using_spec": False, "sample_rate": SR, "use_soundfile": False}
        arch = {"hop_length": cfg.hop_length, "segment_size": cfg.segment_size, "overlap": cfg.overlap, "batch_size": a.batch, "enable_denoise": False,
                "b200_precision": a.precision, "b200_sharded": ctx.world > 1}
        self.plugin = MDXSeparator(common_config=common, arch_config=arch)
        os.unlink(path)
        self.eng, self.net = self.plugin.engine, self.plugin.net
        mix = music(self.N, 1234)
        if ctx.world > 1:
            self.mix_host = ctx.shared_host("mix", (2, self.N))
            if ctx.rank == 0:
                self.mix_host.numpy()[...] = mix
            self.out_host = [ctx.shared_host(f"out{i}", (self.N, 2)) for i in range(2)]
            ctx.barrier()
        else:
            self.mix_host = torch.from_numpy(mix).pin_memory()
        self.mix_dev = self.mix_host.cuda(non_blocking=True)
        torch.cuda.synchronize()
        self.h2d = self.d2h = 0

    def step_device(self):
        return self.eng.separate_device(self.mix_dev, 0.9, 0.0)

    def outputs(self, result):
        p, s = result  # (N, 2) each
        return {"primary": p.T, "secondary": s.T}

    def step_e2e(self):
        if self.ctx.world > 1:
            self.h2d, self.d2h = self.plugin.separate_host_shared(self.mix_host, self.out_host[0], self.out_host[1])
        else:
            p, s = self.plugin.separate_host(self.mix_host)
            self.h2d, self.d2h = self.mix_host.numel() * 4, (p.size + s.size) * 4

    def roofline(self, peaks):
        net, a = self.net, self.args
        net.profile(True)
        self.step_device()
        self.ctx.torch.cuda.synchronize()
        prof = net.profile_read()
        net.profile(False)
        net_ms = sum(v["ms"] for v in prof.values())
        # dominant kernel = the single launch SHAPE with the most device time: the 3x3 convolutions at U-Net scale 0 (one shape, 2 launches per block)
        tname, tv = ("conv3x3_scale0", prof["conv3x3_scale0"]) if prof.get("conv3x3_scale0", {}).get("ms", 0) > 0 else max(prof.items(), key=lambda kv: kv[1]["ms"])
        tf = tv["flops"] / (tv["ms"] * 1e-3) / 1e12 if tv["ms"] > 0 else 0.0
        kname = f"umma_conv3_kernel<48>[{tname}]" if a.precision else f"conv2d_simt_kernel[{tname}]"
        traffic, tsrc = ncu_traffic(f"{tname}_b{a.batch}_p{a.precision}")
        return {
            "kernel": kname, "bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"], "traffic": traffic,
            "traffic_source": tsrc, "peak_source": peaks["source"],
            "arithmetic": "bf16x3 split (3 tcgen05 MMAs per algorithmic MAC): attainable = peak/3" if a.precision else "fp32 FMA (no tensor cores)",
            "frac_of_attainable": (3.0 if a.precision else 1.0) * tf / peaks["bf16_tflops"],
            "launches": tv["launches"], "avg_launch_ms": tv["ms"] / max(1, tv["launches"]),
            "algorithmic_flops_per_launch": tv["flops"] / max(1, tv["launches"]), "algorithmic_bytes_per_launch": tv["bytes"] / max(1, tv["launches"]),
            "hbm_view": {"achieved_gbs": tv["bytes"] / (tv["ms"] * 1e-3) / 1e9 if tv["ms"] > 0 else 0.0, "peak_gbs": peaks["hbm_gbs"]},
            "share_of_net_time": tv["ms"] / max(1e-9, net_ms), "net_ms_per_step": net_ms,
            "by_category_ms": {k: round(v["ms"], 3) for k, v in prof.items() if v["launches"]},
            "by_category_tflops": {k: round(v["flops"] / (v["ms"] * 1e-3) / 1e12, 1) for k, v in prof.items() if v["ms"] > 0 and v["flops"] > 0},
        }

    def parity(self):
        ctx, torch = self.ctx, self.ctx.torch
        from audio_separator.separator.b200 import engine, mdx_weights

        cfg = self.cfg
        if ctx.world > 1:
            got = self.step_device()  # every rank takes part
            out = None
            if ctx.rank == 0:
                single = engine.MdxEngine(self.net, cfg.n_fft, cfg.hop_length, cfg.dim_f, cfg.segment_size, cfg.overlap, cfg.compensate, batch_size=self.args.batch)
                ref = single.separate_device(self.mix_dev, 0.9, 0.0)
                diff = max(float((g - r).abs().max()) for g, r in zip(got, ref))
                # the end-to-end path wrote the shared host buffers: same numbers again
                hd = max(float((h.cuda() - r).abs().max()) for h, r in zip(self.out_host, ref))
                out = {"kind": f"time-sharded x{ctx.world} (NCCL halo + gather) vs single-GPU run of the same engine, whole {self.minutes:g}-min track, both stems",
                       "bit_identical": bool(all(torch.equal(g, r) for g, r in zip(got, ref))), "max_abs_diff": diff, "e2e_host_buffers_max_abs_diff": hd, "gate": 1e-4}
            ctx.barrier()
            return out
        n = min(self.N, 10 * SR)  # BASELINE configs[0]: 10 s = 3 chunks
        hp = mdx_weights.infer_hparams_from_state(self.w)
        ref_net = engine.MdxNet(mdx_weights.flatten_state(self.w, **hp), dim_t=cfg.dim_t, max_batch=1, precision=0, **hp)
        ref_eng = engine.MdxEngine(ref_net, cfg.n_fft, cfg.hop_length, cfg.dim_f, cfg.segment_size, cfg.overlap, cfg.compensate)
        x = self.mix_dev[:, :n].contiguous()
        got, ref = self.eng.separate_device(x, 0.9, 0.0), ref_eng.separate_device(x, 0.9, 0.0)
        diff = max(float((g - r).abs().max()) for g, r in zip(got, ref))
        p, s = self.plugin.separate_host(self.mix_host)
        full = self.step_device()
        same = bool(torch.equal(torch.from_numpy(p).cuda(), full[0]) and torch.equal(torch.from_numpy(s).cuda(), full[1]))
        return {"kind": "tcgen05 bf16x3 path vs the fp32 SIMT path of the same library, 10-s excerpt (3 chunks, full-size net), both stems; the oracle comparison is tests/test_mdx_gpu.py",
                "max_abs_diff": diff, "gate": 1e-4, "e2e_equals_device_resident": same}

    # ---- CPU arm: chunks [3i, 3i+3) of the SAME 68-chunk grid per step (run_model + window + accumulate, as the reference's demix loop does)
    def cpu_setup(self):
        import mdx_oracle as O

        self.O = O
        self.cfg = O.MDXConfig()
        self.cpu_mix = O.normalize(music(self.N, 1234), 0.9, 0.0)
        self.cpu_w = O.make_convtdfnet_weights(self.cfg, seed=11, out_gain=MDX_OUT_GAIN)
        self.cores = pick_cpu_threads(lambda: O.convtdfnet_forward(self.cpu_w, self.cfg, __import__("numpy").zeros((1, 4, self.cfg.dim_f, self.cfg.dim_t), "float32")))
        _, _, starts = O.chunk_starts(self.N, self.cfg)
        self.n_chunks = len(starts)

    def cpu_step(self, i, k=3):
        O = self.O
        idx = [(3 * i + j) % self.n_chunks for j in range(k)]
        t0 = time.perf_counter()
        O.demix(self.cpu_mix, self.cfg, lambda s: O.convtdfnet_forward(self.cpu_w, self.cfg, s), only_chunks=idx)
        wall = time.perf_counter() - t0
        return self.audio_seconds * k / self.n_chunks, wall  # audio-seconds these chunks stand for in the whole-track grid

    def cpu_sample_text(self, k=3):
        return (f"{k} of the {self.n_chunks} chunks of the same {self.minutes:g}-min grid per step (rotating), STFT -> torch-CPU fp32 ConvTDFNet -> iSTFT -> window/accumulate "
                "(oracle/mdx_oracle.py); RTF = (track seconds x k/68) / wall; reference package not installable offline (onnxruntime, librosa wheels absent)")


# ======================================================================================================== htdemucs_ft
class DemucsWorkload:
    name = "htdemucs_ft"
    FLOPS_PER_FORWARD = 334.9e9  # SURVEY.md section 8d, measured by forward hooks on the reference module

    def __init__(self, args):
        self.args = args
        self.minutes = args.minutes or 5.0
        self.N = int(self.minutes * 60 * SR)
        self.audio_seconds = self.N / SR
        self.batch = args.demucs_batch

    def config(self):
        return {"workload": f"htdemucs_ft geometry (bag of 4 HTDemucs, 48 ch, depth 4, 5-layer 512-d cross-transformer, one-hot bag weights), {self.minutes:g}-min 44.1 kHz stereo synthetic, "
                            "shifts=2, overlap=0.25, segment 7.8 s", "segments_per_forward": self.batch, "l2": "inputs larger than L2 (106 MB track, 424 MB of stems, > 1 GB activations per forward)",
                "parallelism": f"time-sharded segments x{self.args.gpus}" if self.args.gpus > 1 else "single GPU"}

    def setup(self, ctx):
        import random

        import demucs_oracle as D
        from audio_separator.separator.b200 import demucs as dm

        torch = ctx.torch
        self.ctx, self.D, self.dm = ctx, D, dm
        self.ocfg = D.HTConfig()
        self.nets = [dm.HTDemucsNet(dm.HTDemucsConfig(), D.make_weights(self.ocfg, seed=11 + i), device=torch.device("cuda", ctx.local)) for i in range(4)]
        self.bag = [[1.0 if s == m else 0.0 for s in range(4)] for m in range(4)]  # htdemucs_ft.yaml: one fine-tuned model per source
        self.eng = dm.DemucsEngine(self.nets, bag_weights=self.bag, overlap=0.25, batch_size=self.batch, dist=ctx.dist)
        rng = random.Random(0)
        self.offsets = [[rng.randint(0, SR // 2) for _ in range(2)] for _ in self.nets]  # the randint draws of apply.py:207, fixed
        mix = music(self.N, 1235)
        if ctx.world > 1:
            self.mix_host = ctx.shared_host("dmix", (2, self.N))
            if ctx.rank == 0:
                self.mix_host.numpy()[...] = mix
            self.out_host = ctx.shared_host("dout", (4, 2, self.N))
            ctx.barrier()
        else:
            self.mix_host = torch.from_numpy(mix).pin_memory()
            self.out_host = torch.empty((4, 2, self.N), dtype=torch.float32).pin_memory()
        self.mix_dev = self.mix_host.cuda(non_blocking=True)
        torch.cuda.synchronize()
        seg, stride = self.ocfg.seg_len, int(0.75 * self.ocfg.seg_len)
        self.n_forwards = sum(len(range(0, self.N + SR // 2 - o, stride)) for offs in self.offsets for o in offs)
        self.h2d = self.d2h = 0

    def step_device(self):
        part = self.eng.demix_device(self.mix_dev, self.offsets)
        return self.eng.gather(part, self.N)

    def outputs(self, result):
        return {"sources": result}  # (4, 2, N)

    def step_e2e(self):
        self.h2d, self.d2h = self.eng.demix_host(self.mix_host, self.out_host, self.offsets)

    def roofline(self, peaks, ms_step=None):
        tf = self.n_forwards * self.FLOPS_PER_FORWARD / (ms_step * 1e-3) / 1e12 * 1.0 / max(1, self.ctx.world) if ms_step else 0.0
        return {"kernel": "HTDemucs forward (every launch of the graph: tc_f32_kernel GEMM / conv, fused DConv, attention, norms, STFT / iSTFT)", "bound": "tensor",
                "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": tf / peaks["bf16_tflops"], "traffic": None, "peak_source": peaks["source"],
                "arithmetic": "bf16x3 split inside the GEMM / conv kernels: attainable = peak/3", "frac_of_attainable": 3.0 * tf / peaks["bf16_tflops"],
                "forwards_per_step": self.n_forwards, "algorithmic_flops_per_forward": self.FLOPS_PER_FORWARD, "per_gpu": True,
                "note": "whole-forward figure (algorithmic flops of all forwards / step time / GPUs); per-kernel launch list: profiles/r02_htdemucs_launches_b4.txt"}

    def parity(self):
        ctx, torch = self.ctx, self.ctx.torch
        if ctx.world == 1:
            return {"kind": "single GPU: parity against the reference goldens and the oracle is tests/test_demucs_gpu.py (incl. one full-size segment)", "gate": 1e-4}
        got = self.step_device()
        out = None
        if ctx.rank == 0:
            single = self.dm.DemucsEngine(self.nets, bag_weights=self.bag, overlap=0.25, batch_size=self.batch)
            ref = single.demix_device(self.mix_dev, self.offsets)
            out = {"kind": f"time-sharded x{ctx.world} (NCCL halo + gather) vs single-GPU run of the same engine, whole {self.minutes:g}-min track, 4 sources",
                   "bit_identical": bool(torch.equal(got, ref)), "max_abs_diff": float((got - ref).abs().max()), "e2e_host_buffers_max_abs_diff": float((self.out_host.cuda() - ref).abs().max()), "gate": 1e-4}
        ctx.barrier()
        return out

    def cpu_setup(self):
        import demucs_oracle as D

        self.D = D
        self.ocfg = D.HTConfig()
        self.cpu_w = D.make_weights(self.ocfg, seed=11)
        self.cpu_seg = music(self.ocfg.seg_len, 1235)[None]
        self.cores = pick_cpu_threads(lambda: D.forward(self.cpu_w, self.ocfg, self.cpu_seg))
        stride = int(0.75 * self.ocfg.seg_len)
        self.n_forwards = 8 * len(range(0, self.N + SR // 4, stride))

    def cpu_step(self, i, k=1):
        t0 = time.perf_counter()
        for _ in range(k):
            self.D.forward(self.cpu_w, self.ocfg, self.cpu_seg)
        return self.audio_seconds * k / self.n_forwards, time.perf_counter() - t0

    def cpu_sample_text(self, k=1):
        return f"{k} of the {self.n_forwards} segment forwards of the same workload per step (torch-CPU fp32 HTDemucs, oracle/demucs_oracle.py); RTF = (track seconds x k/{self.n_forwards}) / wall"


# ======================================================================================================== MDX23C
class MdxcWorkload:
    name = "mdx23c"
    FLOPS_PER_CHUNK = 2434.1e9

    def __init__(self, args):
        self.args = args
        self.minutes = args.minutes or 10.0
        self.N = int(self.minutes * 60 * SR)
        self.audio_seconds = self.N / SR

    def config(self):
        return {"workload": f"MDX23C-8KFFT-InstVoc_HQ topology (TFC_TDF_net, n_fft 8192, dim_f 4096, 5 scales, 128..768 channels), {self.minutes:g}-min 44.1 kHz stereo synthetic, overlap=8, dim_t 256",
                "chunks_per_forward": 2, "l2": "inputs larger than L2", "parallelism": f"time-sharded chunks x{self.args.gpus}" if self.args.gpus > 1 else "single GPU"}

    def setup(self, ctx):
        import mdxc_oracle as X
        from audio_separator.separator.b200 import engine

        torch = ctx.torch
        self.ctx, self.X, self.engine = ctx, X, engine
        self.cfg = cfg = X.MDXCConfig()
        self.w = X.make_weights(cfg, seed=1, out_gain=0.3)
        self.net = engine.TfcNet(self.w, cfg.dim_f, cfg.dim_t, cfg.num_subbands, 2, cfg.num_scales, cfg.num_blocks_per_scale, cfg.num_channels_model, cfg.growth, cfg.bottleneck_factor, cfg.num_targets, max_batch=2)
        self.eng = engine.MdxcEngine(self.net, cfg.n_fft, cfg.hop_length, cfg.dim_f, cfg.dim_t, cfg.overlap, dist=ctx.dist)
        import mdx_oracle as O

        mix = O.normalize(music(self.N, 1236), 0.9, 0.0)
        self.mix_host = torch.from_numpy(mix).pin_memory()
        self.out_host = torch.empty((cfg.num_targets, 2, self.N), dtype=torch.float32).pin_memory() if ctx.rank == 0 else None
        self.mix_dev = self.mix_host.cuda(non_blocking=True)
        torch.cuda.synchronize()
        self.n_chunks = self.eng.grid(self.N)[3]
        self.h2d = self.d2h = 0

    def step_device(self):
        return self.eng.gather(self.eng.demix_device(self.mix_dev), self.N)

    def outputs(self, result):
        return {"stems": result}  # (num_targets, 2, N)

    def step_e2e(self):
        d = self.mix_host.cuda(non_blocking=True)
        full = self.eng.gather(self.eng.demix_device(d), self.N)
        if full is not None:
            self.out_host.copy_(full, non_blocking=True)
        self.ctx.torch.cuda.current_stream().synchronize()
        self.h2d, self.d2h = self.mix_host.numel() * 4, (self.out_host.numel() * 4 if full is not None else 0)

    def roofline(self, peaks, ms_step=None):
        tf = self.n_chunks * self.FLOPS_PER_CHUNK / (ms_step * 1e-3) / 1e12 / max(1, self.ctx.world) if ms_step else 0.0
        return {"kernel": "TFC_TDF_net forward (umma_conv3_kernel / umma_pair_kernel launches of one chunk)", "bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": tf / peaks["bf16_tflops"], "traffic": None, "peak_source": peaks["source"], "arithmetic": "bf16x3 split: attainable = peak/3",
                "frac_of_attainable": 3.0 * tf / peaks["bf16_tflops"], "chunks_per_step": self.n_chunks, "algorithmic_flops_per_chunk": self.FLOPS_PER_CHUNK, "per_gpu": True}

    def parity(self):
        ctx, torch = self.ctx, self.ctx.torch
        if ctx.world == 1:
            return {"kind": "single GPU: parity against the reference goldens and the oracle is tests/test_mdxc_gpu.py", "gate": 1e-4}
        got = self.step_device()
        out = None
        if ctx.rank == 0:
            cfg = self.cfg
            single = self.engine.MdxcEngine(self.net, cfg.n_fft, cfg.hop_length, cfg.dim_f, cfg.dim_t, cfg.overlap)
            n = min(self.N, 60 * SR)  # the first minute on one GPU (818 chunks would take the whole bench budget)
            ref = single.demix_device(self.mix_dev[:, :n].contiguous())
            m = n - single.chunk_size  # samples whose covering chunks see the same audio in both runs
            out = {"kind": f"time-sharded x{ctx.world} (NCCL halo + gather) vs single-GPU run of the same engine on the first {n / SR:g} s (compared where the chunk supports coincide)",
                   "bit_identical": bool(torch.equal(got[..., :m], ref[..., :m])), "max_abs_diff": float((got[..., :m] - ref[..., :m]).abs().max()), "gate": 1e-4}
        ctx.barrier()
        return out

    def cpu_setup(self):
        import mdxc_oracle as X

        self.X = X
        self.cfg = X.MDXCConfig()
        self.cpu_w = X.make_weights(self.cfg, seed=1, out_gain=0.3)
        self.cpu_chunk = music(self.cfg.chunk_size, 1236)[None]
        self.cores = pick_cpu_threads(lambda: X.net_forward(self.cpu_w, self.cfg, self.cpu_chunk))
        self.n_chunks = X.chunk_grid(self.N, self.cfg)[3]

    def cpu_step(self, i, k=1):
        t0 = time.perf_counter()
        for _ in range(k):
            self.X.net_forward(self.cpu_w, self.cfg, self.cpu_chunk)
        return self.audio_seconds * k / self.n_chunks, time.perf_counter() - t0

    def cpu_sample_text(self, k=1):
        return f"{k} of the {self.n_chunks} chunk forwards of the same workload per step (torch-CPU fp32 TFC_TDF_net incl. STFT / iSTFT, oracle/mdxc_oracle.py)"


# ======================================================================================================== VR batch
class VrWorkload:
    name = "vr"
    FLOPS_PER_PATCH = 2363.4e9

    def __init__(self, args):
        self.args = args
        self.minutes = args.minutes or 3.0
        self.tracks = args.tracks
        self.N = int(self.minutes * 60 * SR)
        self.audio_seconds = self.tracks * self.N / SR

    def config(self):
        return {"workload": f"9_HP2-UVR geometry (CascadedASPPNet 537238, 4band_v2, window 512, aggression 10), batch of {self.tracks} x {self.minutes:g}-min 44.1 kHz stereo synthetic tracks",
                "patches_per_forward": 4, "l2": "inputs larger than L2", "parallelism": f"whole tracks round-robin over {self.args.gpus} GPUs, no collective" if self.args.gpus > 1 else "single GPU"}

    def setup(self, ctx):
        import mdx_oracle as O
        import vr_oracle as V
        from audio_separator.separator.b200 import vr

        torch = ctx.torch
        self.ctx = ctx
        arch = 537238
        self.eng = vr.VREngine(vr.VRNet(arch, 1344, V.make_weights(arch, seed=9), device=torch.device("cuda", ctx.local)), V.four_band_v2_param(), window_size=512, aggression=10, batch_size=4)
        self.mine = list(range(ctx.rank, self.tracks, ctx.world))  # vr_separator.py has no cross-file state: tracks are independent units
        base = O.normalize(music(self.N, 1234), 0.9, 0.0)
        # distinct tracks from one synthesised pattern: rotate it by a track-dependent offset (cheap, deterministic)
        self.host = [torch.from_numpy(__import__("numpy").roll(base, 7919 * (t + 1), axis=1).copy()).pin_memory() for t in self.mine]
        self.dev = [h.cuda() for h in self.host]
        torch.cuda.synchronize()
        self.h2d = self.d2h = 0
        self.patches = None

    def step_device(self):
        out = []
        for d in self.dev:
            spec = self.eng.loading_mix(d)
            y, v = self.eng.inference(spec)
            out.append((self.eng.spec_to_wav(y), self.eng.spec_to_wav(v)))
        return out

    def outputs(self, result):
        """This rank's tracks: primary and secondary (2, M) of each."""
        return {f"track{t}_{stem}": w for t, pair in zip(self.mine, result) for stem, w in zip(("primary", "secondary"), pair)}

    def step_e2e(self):
        h2d = d2h = 0
        for h in self.host:
            p, s = self.eng.separate(h.numpy())
            h2d += h.numel() * 4
            d2h += (p.size + s.size) * 4
        self.h2d, self.d2h = h2d, d2h

    def roofline(self, peaks, ms_step=None):
        frames = self.N // 480 + 1
        patches = self.tracks * (-(-frames // 256))
        tf = patches * self.FLOPS_PER_PATCH / (ms_step * 1e-3) / 1e12 / max(1, self.ctx.world) if ms_step else 0.0
        return {"kernel": "CascadedASPPNet.predict_mask (tc_f32_kernel convolutions of one patch batch)", "bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                "frac": tf / peaks["bf16_tflops"], "traffic": None, "peak_source": peaks["source"], "arithmetic": "bf16x3 split: attainable = peak/3",
                "frac_of_attainable": 3.0 * tf / peaks["bf16_tflops"], "patches_per_step": patches, "algorithmic_flops_per_patch": self.FLOPS_PER_PATCH, "per_gpu": True}

    def parity(self):
        return {"kind": "whole tracks are independent units (no cross-rank arithmetic): parity is the single-GPU suite tests/test_vr_gpu.py", "gate": 1e-4,
                "note": "multi-band synthesis up-sampling (libsamplerate sinc_fastest) is a Kaiser polyphase stand-in: parity unpinned for that step (DESIGN.md section 11)"}

    def cpu_setup(self):
        import numpy as np

        import vr_oracle as V

        self.V = V
        arch = 537238
        self.cpu_w = V.make_weights(arch, seed=9)
        self.cpu_cfg = V.VRConfig(param=V.four_band_v2_param(), nn_architecture=arch)
        self.cpu_x = np.abs(np.random.default_rng(0).standard_normal((1, 2, 673, 512))).astype(np.float32)
        self.cores = pick_cpu_threads(lambda: V.predict_mask(self.cpu_w, self.cpu_cfg, self.cpu_x))
        self.patches = self.tracks * (-(-(self.N // 480 + 1) // 256))

    def cpu_step(self, i, k=1):
        t0 = time.perf_counter()
        for _ in range(k):
            self.V.predict_mask(self.cpu_w, self.cpu_cfg, self.cpu_x)
        return self.audio_seconds * k / self.patches, time.perf_counter() - t0

    def cpu_sample_text(self, k=1):
        return f"{k} of the {self.patches} patch forwards of the same workload per step (torch-CPU fp32 CascadedASPPNet, oracle/vr_oracle.py; STFT front / back end not included)"


WORKLOADS = {"mdx": MdxWorkload, "htdemucs_ft": DemucsWorkload, "mdx23c": MdxcWorkload, "vr": VrWorkload}

_CPU_THREADS = {}


def pick_cpu_threads(one_forward):
    """All host threads the CPU path can use PRODUCTIVELY: torch-CPU convolutions stop scaling (and regress) well before 128 threads, so time one
    network forward at a few thread counts and keep the fastest (reported as `cores`)."""
    import torch

    n = os.cpu_count() or 1
    cands = sorted({n, max(1, n // 2), min(n, 32), min(n, 16)}, reverse=True)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        one_forward()
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    return best


def cpu_leg(wl, steps, k=None):
    """`steps` bounded samples of the workload on the host cores -> (rtf, cores, wall_per_step, sample text)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    wl.cpu_setup()
    kw = {} if k is None else {"k": k}
    secs = wall = 0.0
    for i in range(steps):
        s, w = wl.cpu_step(i, **kw)
        secs += s
        wall += w
    return secs / wall, wl.cores, wall / steps, wl.cpu_sample_text(**kw)


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    wl = WORKLOADS[args.workload](args)
    value, cores, wall, sample = cpu_leg(wl, max(1, args.steps))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "x realtime", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": wall * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": wl.config(),
        "cpu_baseline": {"value": value, "unit": "x realtime", "cores": cores, "host_cpus": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "x realtime", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def measure(wl, ctx, args, steps, warmup, with_cpu, dump_bytes=DUMP_BYTES):
    """One workload on this rank set -> the JSON line (rank 0) or None.  With --dump-outputs, rank 0 writes what the last timed step returned."""
    from audio_separator.separator.b200 import _lib

    wl.setup(ctx)
    ms_step = 0.0
    sampler = ClockSampler(ctx.local)
    for _ in range(warmup):
        wl.step_device()
    ctx.barrier()
    if ctx.rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    ms_step, last = ctx.timed(wl.step_device, steps, 0)
    launches = ctx.sum_over_ranks(_lib.launch_count() - launches0)[0]
    clocks = sampler.summary() if ctx.rank == 0 else None
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, wl.name, wl.outputs(last), dump_bytes)
    del last
    ms_e2e, _ = ctx.timed(wl.step_e2e, steps, 1)
    h2d, d2h = ctx.sum_over_ranks(wl.h2d, wl.d2h)
    peaks = load_peaks()
    roof = wl.roofline(peaks) if isinstance(wl, MdxWorkload) else wl.roofline(peaks, ms_step)
    parity = None if args.no_parity else wl.parity()
    if ctx.rank != 0:
        return None
    cpu_b = None
    if with_cpu:
        rtf, cores, wall, sample = cpu_leg(wl, 1)
        cpu_b = {"value": rtf, "unit": "x realtime", "cores": cores, "kind": "port", "sample": sample + f" ({wall:.1f} s CPU wall)"}
    return {
        "metric": METRIC, "value": wl.audio_seconds / (ms_step * 1e-3), "unit": "x realtime", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": wl.config(),
        "e2e": {"value": wl.audio_seconds / (ms_e2e * 1e-3), "unit": "x realtime", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "entry": "plugin-level host-buffer call (MDXSeparator.separate_host / separate_host_shared, DemucsEngine.demix_host, ...): pinned input uploaded, stems downloaded, inside the timed region"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "parity": parity, "cpu_baseline": cpu_b,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="mdx", choices=sorted(WORKLOADS))
    ap.add_argument("--also", default="htdemucs_ft", help="second workload measured by the default (mdx) run and reported under \"also\" (none = skip)")
    ap.add_argument("--minutes", type=float, default=None, help="track length (default: the BASELINE config's)")
    ap.add_argument("--batch", type=int, default=None, help="MDX chunks per network forward (default 8; with N > 1 all the chunks of a rank, up to 12)")
    ap.add_argument("--demucs-batch", type=int, default=13, help="HTDemucs segments per forward")
    ap.add_argument("--tracks", type=int, default=32, help="VR workload: tracks in the batch")
    ap.add_argument("--precision", type=int, default=1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<workload>_<name>.npy (float32; a fixed seeded sample of time positions, under 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.batch is None:
        args.batch = 8 if args.gpus == 1 else min(12, -(-68 // args.gpus))  # 8 chunks per forward measured 2 % faster than 4 on one box (1242 vs 1215)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))  # synthetic weights + programme material generators, and the cpu legs
    if args.impl == "reference":
        return run_reference(args)
    ctx = Ctx(args)
    warmup = max(args.warmup, 3)
    with_also = args.workload == "mdx" and args.also in WORKLOADS and args.also != "mdx"
    dump_bytes = DUMP_BYTES // 2 if with_also else DUMP_BYTES
    line = measure(WORKLOADS[args.workload](args), ctx, args, args.steps, warmup, with_cpu=not args.no_cpu_baseline, dump_bytes=dump_bytes)
    if with_also:
        import gc
        import signal

        printed = []

        def emit(extra):
            if line is not None and not printed:
                printed.append(1)
                line["also"] = {args.also: extra}
                print(json.dumps(line), flush=True)

        # the headline line is already measured: a failure of the second workload (here or on a peer rank -- torchrun then SIGTERMs this one) must not lose it
        signal.signal(signal.SIGTERM, lambda *_: (emit({"error": "terminated: a peer rank failed during this workload"}), os._exit(0)))
        gc.collect()
        ctx.torch.cuda.empty_cache()
        try:
            extra = measure(WORKLOADS[args.also](args), ctx, args, args.steps, 3, with_cpu=not args.no_cpu_baseline, dump_bytes=dump_bytes)
        except Exception as e:  # noqa: BLE001
            import traceback

            extra = {"error": f"{type(e).__name__}: {e}"[:500], "where": [ln.strip()[:160] for ln in traceback.format_exc().splitlines() if ln.strip().startswith("File")][-6:]}
            traceback.print_exc()
            emit(extra)
            os._exit(0 if ctx.rank == 0 else 1)
        emit(extra)
    elif line is not None:
        print(json.dumps(line), flush=True)
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
