"""Timing of Flow.log_prob_grad (csrc/flow_grad.cu) and of one nll_grad refinement step (eval.py:464-480), fused vs composed autograd.

    python tools/grad_bench.py --out grad_bench.json

CUDA events around each call, median of --reps timed calls after --warmup untimed ones.  Flow: the symsol settings at F = 2048
(seeded weights).  log_prob_grad at N = 256, 4096 and 1 048 576 rows (64 images, image-major); one refinement step
(quaternion -> matrix, flow + gradient, backward, Adam) at B = 32, 256 and 1024 rows, once with the fused kernel and once with
autograd through the per-layer operators (flow(R.requires_grad_(), rows) + backward)."""
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
from rotationnormflow_b200 import evalpath  # noqa: E402


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
    return statistics.median(ts), min(ts), max(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "grad_bench measures on the GPU"
    dev = torch.device("cuda", 0)
    cfg = rnf.load_config("symsol", feature_dim=2048)
    torch.manual_seed(0)
    np.random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        flow = rnf.get_flow(cfg).to(dev).eval()
    F = flow.feature_dim
    gen = torch.Generator(device=dev).manual_seed(1)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        smi = "nvidia-smi not found"
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi, config="symsol", F=F, layers=len(flow.layers),
               warmup=args.warmup, reps=args.reps, log_prob_grad=[], refine_step=[])

    def rand_rot(n):
        q = torch.randn(n, 4, device=dev, generator=gen)
        return evalpath.quaternion_to_matrix(q / q.norm(dim=-1, keepdim=True))

    for N in (256, 4096, 1 << 20):
        B = 64
        R = rand_rot(N)
        feat = torch.relu(torch.randn(B, F, device=dev, generator=gen))
        med, lo, hi = timed(lambda: flow.log_prob_grad(R, feat), args.warmup, args.reps)
        res["log_prob_grad"].append(dict(N=N, images=B, ms_median=med, ms_min=lo, ms_max=hi, rows_per_s=N / (med * 1e-3)))
        print(res["log_prob_grad"][-1], flush=True)

    for B in (32, 256, 1024):
        feat = torch.relu(torch.randn(B, F, device=dev, generator=gen))
        q0 = evalpath.matrix_to_quaternion(rand_rot(B))
        for path in ("fused", "composed"):
            q = q0.clone().requires_grad_(True)
            opt = torch.optim.Adam([q], lr=1e-3)

            def step():
                with torch.enable_grad():
                    R = evalpath.quaternion_to_matrix(q / q.norm(dim=-1, keepdim=True))
                    opt.zero_grad()
                    if path == "fused":
                        _, G = flow.log_prob_grad(R.detach(), feat)
                        R.backward(-G)
                    else:
                        _, ldj = flow(R, feat)                  # R requires grad: per-layer operators of train.py
                        (-ldj.sum()).backward()
                    opt.step()

            med, lo, hi = timed(step, args.warmup, args.reps)
            res["refine_step"].append(dict(B=B, path=path, ms_median=med, ms_min=lo, ms_max=hi))
            print(res["refine_step"][-1], flush=True)
    for B in (32, 256, 1024):
        f, c = [r["ms_median"] for r in res["refine_step"] if r["B"] == B]
        res.setdefault("speedup_fused_over_composed", {})[str(B)] = c / f
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res["speedup_fused_over_composed"]))


if __name__ == "__main__":
    main()
