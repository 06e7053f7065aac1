"""Strong scaling of ONE 5-minute track through the time-sharded BS-Roformer engine (measurement tool).

    python -m torch.distributed.run --nproc-per-node N tests/dev/roformer_sharded_bench.py [--steps 2] [--warmup 1] [--minutes 5]

model_bs_roformer_ep_317 geometry (dim 512, depth 12, 62 bands, n_fft 2048 / hop 441, dim_t 801, overlap 8 -> step = chunk), 2 chunks per forward,
seeded synthetic weights and mix.  The mix is resident in HBM on every rank; one step = RoformerEngine(dist=).demix_device + gather to rank 0, timed
with CUDA events on rank 0 after a barrier.  Rank 0 prints one JSON line: RTF, units / forwards per rank, parity against a single-GPU run of the plain
engine on rank 0, and the GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [os.path.join(ROOT, "python-audio-separator_b200"), os.path.join(ROOT, "oracle")]
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

SR = 44100


def gpu_info(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(index)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--minutes", type=float, default=5.0)
    a = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()

    import mdx_oracle as M
    import roformer_oracle as R
    from audio_separator.separator.b200 import roformer as rf
    from audio_separator.separator.b200.sharded import balanced_batches, plan_start_shards

    kw = dict(stft_hop_length=441)
    net = rf.BSRoformerNet(rf.BSRoformerConfig(**kw), R.make_weights(R.BSRoformerConfig(**kw), seed=8))
    eng = rf.RoformerEngine(net, 801, 8, SR, n_instruments=2, batch_size=2, dist=dist)
    secs = a.minutes * 60
    mix = M.normalize(M.synth_music(int(secs * SR), seed=5), 0.9, 0.0)
    md = torch.from_numpy(mix).cuda()
    N = md.shape[1]
    starts = eng.chunk_starts(N)
    shards = plan_start_shards(N, world, starts, eng.chunk_size)

    def step():
        return eng.gather(eng.demix_device(md), N)

    for _ in range(a.warmup):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        full = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    info = [None] * world
    dist.all_gather_object(info, gpu_info(local))
    if rank == 0:
        ref = rf.RoformerEngine(net, 801, 8, SR, n_instruments=2, batch_size=2).demix_device(md)
        out = {"metric": "real-time factor (audio-sec/wall-sec) @44.1kHz stereo", "arch": "MDXC/BS-Roformer, time-sharded", "value": round(secs / (ms / 1e3), 1), "unit": "x realtime",
               "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": round(ms, 2), "higher_is_better": True,
               "config": {"workload": f"model_bs_roformer_ep_317 geometry (dim 512, depth 12, 62 bands, n_fft 2048 / hop 441, dim_t 801), {a.minutes:g}-min track, overlap 8",
                          "chunks": len(starts), "chunks_per_forward": 2, "timing": "CUDA events on rank 0 around demix_device + gather, mix resident in HBM"},
               "per_rank": [{"rank": s.rank, "units_computed": s.n_own, "halo_units_received": s.halo, "forwards": len(balanced_batches(s.n_own, 2)), "samples": [s.q0, s.q1]}
                            for s in shards],
               "parity": {"vs": "plain RoformerEngine on one GPU", "bit_identical": bool(torch.equal(full, ref)), "max_abs_diff": float((full - ref).abs().max())},
               "gpus": info}
        print(json.dumps(out), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
