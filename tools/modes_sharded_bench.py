"""Timing of the sharded separated modes (dist.sharded_rotation_modes, csrc/modes.cu rnf_rotation_modes_shard_*) against the grid pass
they follow, on the bench config-5 grid split over the ranks.

    torchrun --nproc_per_node N tools/modes_sharded_bench.py --out profiles/r08_modes_sharded_bench.json

Setup: symsol settings with F = 2048 (random init, seed 0), the 37 748 736-rotation grid of bench config 5 (the level-6 grid under two
offsets, concatenated), split by dist.shard_range, B = 8 images, M = 12 and 60, min_separation 0.35, neighbour_radius the level-6
default.  Each rank materialises its slice of the rotated grid, so the modes see the same rotations the grid pass scores.  CUDA events
around each call, all ranks aligned by a barrier before every timed call, median of --reps after --warmup untimed calls:
  grid         Flow.grid_log_prob(return_logp=True) on the rank's slice: the [B,G_r] log-density the modes are taken from
  modes        sharded_rotation_modes end to end (M + 1 rounds, each rank kernels + one all-gather of B x 80 bytes)
  kernels      the rank's round and merge launches of the same loop, summed per call (events around each)
  collective   the all-gathers of the same loop, summed per call; includes waiting for the slowest rank
  single       (N = 1 only) modes.rotation_modes on the whole grid, and whether the sharded call returned the same bytes
The values (4 B per image and point), labels (1 B) and quaternions (16 B per point) of a rank far exceed the 126 MB L2 at every N
up to 8, so every round streams them from HBM.  The run for N ranks goes into runs[str(N)] of --out (other entries are kept).  GPU
name, power limit and clocks are read in the same run."""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rotationnormflow_b200 as rnf  # noqa: E402
from rotationnormflow_b200 import dist as rdist, evalpath, grid as rgrid  # noqa: E402
from rotationnormflow_b200.modes import RankModes, rotation_modes  # noqa: E402


def barrier(world):
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def timed(fn, warmup, reps, world):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        barrier(world)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return dict(ms_median=statistics.median(ts), ms_min=min(ts), ms_max=max(ts))


def split_modes(lp, rot, lo, M, theta, rho, gather, warmup, reps, world):
    """Rank kernels vs all-gathers of one sharded_rotation_modes call, from events around each launch group."""
    def once():
        ev = []
        rm = RankModes(lp, rot, lo, M, theta, rho)
        for r in range(M + 1):
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            e[0].record()
            rec = rm.propose(r)
            e[1].record()
            g = gather(rec)
            e[2].record()
            rm.merge(r, g)
            e[3].record()
            ev.append(e)
        return ev
    for _ in range(warmup):
        once()
    kern, coll = [], []
    for _ in range(reps):
        barrier(world)
        ev = once()
        torch.cuda.synchronize()
        kern.append(sum(e[0].elapsed_time(e[1]) + e[2].elapsed_time(e[3]) for e in ev))
        coll.append(sum(e[1].elapsed_time(e[2]) for e in ev))
    return dict(kernels_ms_median=statistics.median(kern), collective_ms_median=statistics.median(coll),
                collective_per_round_us=1e3 * statistics.median(coll) / (M + 1))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--images", type=int, default=8)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "modes_sharded_bench measures on the GPU"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    try:
        run(args, world, rank, local, dev)
    finally:
        if world > 1:
            dist.destroy_process_group()


def run(args, world, rank, local, dev):
    cfg = rnf.load_config("symsol", feature_dim=2048)
    torch.manual_seed(0)
    np.random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        flow = rnf.get_flow(cfg).to(dev).eval()
    B, level, n_off = args.images, 6, 2
    gen = torch.Generator().manual_seed(1)
    feat = torch.relu(torch.randn(B, flow.feature_dim, generator=gen)).to(dev)
    offsets = [evalpath._random_rotation(dev, gen) for _ in range(n_off)]
    G1 = 72 * 8 ** level
    G_total = n_off * G1
    lo, hi = rdist.shard_range(G_total, rank, world)
    pieces = []
    for k in range(n_off):                         # this rank's part of copy k: [max(lo, k G1), min(hi, (k+1) G1))
        a, b = max(lo, k * G1), min(hi, (k + 1) * G1)
        if b > a:
            pieces.append(rgrid.healpix_grid(level, a - k * G1, b - k * G1, device=dev) @ offsets[k])
    rot = torch.cat(pieces) if pieces else torch.empty(0, 3, 3, device=dev)
    theta, rho = 0.35, evalpath.default_neighbour_radius(level)
    gather = rdist._record_gather(None)
    res = dict(n_gpus=world, config="bench config 5 grid: symsol F=2048, level 6 x 2 offsets", G_total=G_total, G_rank0=hi - lo if rank == 0 else None,
               images=B, min_separation=theta, neighbour_radius=rho, warmup=args.warmup, reps=args.reps)
    with torch.no_grad():
        res["grid"] = timed(lambda: flow.grid_log_prob(rot, feat, return_logp=True, g_index0=lo), args.warmup, args.reps, world)
        lp = flow.grid_log_prob(rot, feat, return_logp=True, g_index0=lo)["logp"]
        res["modes"] = []
        for M in (12, 60):
            row = dict(M=M, rounds=M + 1, record_bytes_per_gather=B * 80)
            row["sharded"] = timed(lambda: rdist.sharded_rotation_modes(lp, rot, lo, G_total, M, theta, rho), args.warmup, args.reps, world)
            row.update(split_modes(lp, rot, lo, M, theta, rho, gather, args.warmup, args.reps, world))
            row["sharded_over_grid"] = row["sharded"]["ms_median"] / res["grid"]["ms_median"]
            out = rdist.sharded_rotation_modes(lp, rot, lo, G_total, M, theta, rho)
            row["count_mean"] = float(out["count"].float().mean())
            row["local_max_mean"] = float(out["local_max"].float().sum(1).mean())
            if world == 1:
                row["single"] = timed(lambda: rotation_modes(lp, rot, M, theta, rho), args.warmup, args.reps, world)
                ref = rotation_modes(lp, rot, M, theta, rho)
                row["equal_to_rotation_modes"] = all(torch.equal(out[k], ref[k]) for k in ("index", "value", "local_max", "count"))
                row["mass_max_rel_diff"] = float(((out["mass"].double() - ref["mass"].double()).abs()
                                                  / ref["mass"].double().abs().clamp(min=1e-30)).max())
            res["modes"].append(row)
            if rank == 0:
                print("modes", json.dumps(row), flush=True)
    if rank != 0:
        return
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                             capture_output=True, text=True).stdout.strip().splitlines()[:max(world, 1)]
    except OSError:
        smi = ["nvidia-smi not found"]
    res.update(device=torch.cuda.get_device_name(dev), nvidia_smi=smi)
    print("grid", res["grid"], flush=True)
    data = dict(runs={})
    if os.path.exists(args.out):
        with open(args.out) as fh:
            data = json.load(fh)
    data["runs"][str(world)] = res
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(data, fh, indent=1)


if __name__ == "__main__":
    main()
