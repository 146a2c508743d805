"""Timing of the multi-modal pose estimate (csrc/modes.cu, evalpath.estimate_rotation_modes) against the grid pass it follows.

    python tools/modes_bench.py --out profiles/r07_modes_bench.json

Flow: the symsol settings (F = 512, seeded weights), level-5 HEALPix grid (2 359 296 rotations), B = 8 images.  CUDA events
around each call, median of --reps timed calls after --warmup untimed ones:
  grid        Flow.grid_log_prob(return_logp=True): the [B,G] log-density the modes are taken from
  modes       modes.rotation_modes on that log-density, M = 12 and 60 (2M + 3 launches)
  refine      evalpath.refine_rotation on [B,M] seeds (the modes found), 100 Adam steps
  estimate    evalpath.estimate_rotation_modes end to end (grid pass + modes + selection), M = 12, no refinement
The modes rounds stream the values (4 B), labels (1 B) and quaternions (16 B, shared by the images) of every point: at B = 8 that is
132 MB per round, just above the 126 MB L2, so the rounds are timed as they run in the estimate, right after the grid pass wrote the
values.  GPU name, power limit and maximum SM clock are read in the same run."""
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

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rotationnormflow_b200 as rnf  # noqa: E402
from rotationnormflow_b200 import evalpath, grid as rgrid  # noqa: E402
from rotationnormflow_b200.modes import rotation_modes  # noqa: E402


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return dict(ms_median=statistics.median(ts), ms_min=min(ts), ms_max=max(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--level", type=int, default=5)
    ap.add_argument("--images", type=int, default=8)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "modes_bench measures on the GPU"
    dev = torch.device("cuda", 0)
    cfg = rnf.load_config("symsol", feature_dim=512)
    torch.manual_seed(0)
    np.random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        flow = rnf.get_flow(cfg).to(dev).eval()
    F, B = flow.feature_dim, args.images
    gen = torch.Generator().manual_seed(1)
    feat = torch.relu(torch.randn(B, F, generator=gen)).to(dev)
    grid = rgrid.healpix_grid(args.level, device=dev)
    G = grid.shape[0]
    offset = evalpath._random_rotation(dev, gen)
    theta, rho = 0.35, evalpath.default_neighbour_radius(args.level)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        smi = "nvidia-smi not found"
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi, config="symsol", F=F, layers=len(flow.layers), level=args.level,
               G=G, images=B, min_separation=theta, neighbour_radius=rho, warmup=args.warmup, reps=args.reps)
    with torch.no_grad():
        res["grid"] = timed(lambda: flow.grid_log_prob(grid, feat, offset=offset, return_logp=True), args.warmup, args.reps)
        print("grid", res["grid"], flush=True)
        logp = flow.grid_log_prob(grid, feat, offset=offset, return_logp=True)["logp"]
        res["modes"], res["refine"] = [], []
        for M in (12, 60):
            def grid_then_modes():
                lp = flow.grid_log_prob(grid, feat, offset=offset, return_logp=True)["logp"]
                return rotation_modes(lp, grid, M, theta, rho)
            both = timed(grid_then_modes, args.warmup, args.reps)
            alone = timed(lambda: rotation_modes(logp, grid, M, theta, rho), args.warmup, args.reps)
            bytes_round = B * G * 5 + G * 16
            row = dict(M=M, grid_plus_modes=both, modes_alone=alone,
                       modes_over_grid=(both["ms_median"] - res["grid"]["ms_median"]) / res["grid"]["ms_median"],
                       modes_alone_over_grid=alone["ms_median"] / res["grid"]["ms_median"],
                       bytes_per_round=bytes_round, rounds=M + 1,
                       streamed_GB_per_s=(M + 1) * bytes_round / (alone["ms_median"] * 1e-3) / 1e9)
            out = rotation_modes(logp, grid, M, theta, rho)
            row["count_mean"] = float(out["count"].float().mean())
            row["local_max_mean"] = float(out["local_max"].float().sum(1).mean())
            res["modes"].append(row)
            print("modes", row, flush=True)
            seeds = grid[out["index"].clamp(min=0)] @ offset
            r = timed(lambda: evalpath.refine_rotation(flow, feat, seeds, lr=1e-3, steps=100), 1, args.reps)
            res["refine"].append(dict(M=M, steps=100, rows=B * M, **r))
            print("refine", res["refine"][-1], flush=True)
        res["estimate_M12"] = timed(lambda: evalpath.estimate_rotation_modes(flow, feat, 72 * 8 ** args.level, 12, min_separation=theta,
                                                                             offset=offset), args.warmup, args.reps)
        print("estimate", res["estimate_M12"], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps({m["M"]: round(m["modes_alone_over_grid"], 5) for m in res["modes"]}))


if __name__ == "__main__":
    main()
