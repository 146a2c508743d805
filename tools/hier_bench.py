"""Timing and accuracy of the coarse-to-fine grid search (csrc/hgrid.cu, evalpath.estimate_rotation_hierarchical; DESIGN 4.8).

    python tools/hier_bench.py --out profiles/r10_hier_bench.json

Flow: the symsol settings (F = 512, seeded weights), 8 and 1024 images, one fixed offset.  Start level 3; final levels 5, 6, 7, 8;
beam 16, 64, 256.  Per run, CUDA events after --warmup untimed calls, median of --reps:
  coarse      Flow.grid_log_prob(return_logp=True) on the level-3 grid + grid.top_k
  level l     grid.healpix_children + Flow.forward on the 8 x beam children per image + grid.top_k
  total       evalpath.estimate_rotation_hierarchical end to end
plus the rotations scored per image.  Accuracy against the full grid arg-max (Flow.grid_log_prob): at level 5 on all images, at level 6
on 8 images; the log p gap is full max - search log p (0 where the search found the arg-max).  Baselines: the full level-5 pass
(8 and 1024 images) and the level-6 pass (8 images).  GPU name, power limit and maximum SM clock are read in the same run."""
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
    return statistics.median(ts)


def stages(flow, feat, L, l0, beam, offset):
    """The search of estimate_rotation_hierarchical split into its coarse pass and levels, each bracketed by CUDA events."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(L - l0 + 2)]
    ev[0].record()
    lp = flow.grid_log_prob(rgrid.get_closest_available_grid(rgrid.GRID_SIZES[l0], offset.device), feat, offset=offset,
                            return_logp=True)["logp"]
    _, top = rgrid.top_k(lp, None, min(beam, rgrid.GRID_SIZES[l0]))
    ev[1].record()
    for i, level in enumerate(range(l0 + 1, L + 1)):
        ch, rot = rgrid.healpix_children(level - 1, top.reshape(-1), offset)
        n = ch.shape[0] * 8 // feat.shape[0]
        lp = evalpath._score_rows(flow, rot.reshape(-1, 3, 3), feat, n, None, None)
        _, top = rgrid.top_k(lp, ch.reshape(feat.shape[0], n), beam if level == L else min(beam, rgrid.GRID_SIZES[level]))
        ev[i + 2].record()
    ev[-1].synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(len(ev) - 1)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "hier_bench measures on the GPU"
    dev = torch.device("cuda", 0)
    cfg = rnf.load_config("symsol", feature_dim=512)
    torch.manual_seed(0)
    np.random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        flow = rnf.get_flow(cfg).to(dev).eval()
    feats = {B: torch.relu(torch.randn(B, 512, generator=torch.Generator().manual_seed(1))).to(dev) for B in (8, 1024)}
    offset = evalpath._random_rotation(dev, torch.Generator().manual_seed(2))
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()
    except FileNotFoundError:
        smi = "nvidia-smi not found"
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi, config="symsol", F=512, layers=len(flow.layers), start_level=3,
               warmup=args.warmup, reps=args.reps, baselines=[], runs=[])
    full = {}
    with torch.no_grad():
        for B, level, reps in ((8, 5, args.reps), (1024, 5, 1), (8, 6, 1)):
            grid = rgrid.healpix_grid(level)
            ms = timed(lambda: flow.grid_log_prob(grid, feats[B], offset=offset), 1, reps)
            full[(B, level)] = flow.grid_log_prob(grid, feats[B], offset=offset)
            res["baselines"].append(dict(images=B, level=level, rotations_per_image=rgrid.GRID_SIZES[level], grid_pass_ms=ms))
            print(res["baselines"][-1], flush=True)
            del grid
            torch.cuda.empty_cache()
        for B in (8, 1024):
            feat = feats[B]
            for L in (5, 6, 7, 8):
                for beam in (16, 64, 256):
                    Q = rgrid.GRID_SIZES[L]
                    run = lambda: evalpath.estimate_rotation_hierarchical(flow, feat, Q, start_level=3, beam=beam, offset=offset)
                    total = timed(run, args.warmup, args.reps)
                    parts = [stages(flow, feat, L, 3, beam, offset) for _ in range(args.reps)]
                    per = [statistics.median(p[i] for p in parts) for i in range(len(parts[0]))]
                    est, out = run()
                    row = dict(images=B, final_level=L, beam=beam, total_ms=total, coarse_ms=per[0],
                               level_ms={str(3 + i + 1): per[i + 1] for i in range(len(per) - 1)}, evaluated_per_image=out["evaluated"],
                               full_grid_rotations_per_image=Q)
                    if (B, L) in full:
                        f = full[(B, L)]
                        gap = (f["max"] - out["logp"]).double()
                        row.update(agreement_with_full_argmax=(out["index"] == f["argmax"]).double().mean().item(),
                                   logp_gap_max=gap.max().item(), logp_gap_mean=gap.mean().item(),
                                   never_above_full_max=bool((out["logp"] <= f["max"]).all()))
                    res["runs"].append(row)
                    print(row, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
