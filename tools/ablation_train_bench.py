"""Timing of one training step (forward, backward, Adam; agent.py:49-87) of a flow with ablation layers: Flow.forward with autograd
on (train.composed_run: library GEMMs for the conditioners, the rnf_train_* operators of csrc/train_ops.cu for the layers) against
eager torch autograd through the oracle restatement of the reference on the same GPU (OracleFlow(..., torch.float32,
device="cuda").with_grad), the only other implementation of these layers with a backward pass.

    python tools/ablation_train_bench.py --out r05_ablation_train_bench.json

Configuration: settings/modelnet_fisher.yml at full size (24 layers, F = 2080, conditional) with rot = 36Trans (Condition36Trans) and
rot = 9TransLSmith (Condition9Trans); seeded weights and inputs, one image per rotation as agent.py feeds them, loss = -mean(ldj)
(the flow's part of the NLL; the Fisher base term is left out, it is the same for both arms).  CUDA events around each full step,
median of --reps timed steps after --warmup untimed ones; the two arms alternate step by step."""
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
from oracle import rnf_oracle as orc  # noqa: E402


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def run_config(rot, N, dev, warmup, reps):
    cfg = rnf.load_config("modelnet_fisher", rot=rot)
    torch.manual_seed(0)
    np.random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        flow = rnf.get_flow(cfg).to(dev).train()
    F = flow.feature_dim
    oracle = orc.OracleFlow(cfg, flow.state_dict(), torch.float32, device=dev)
    names = [k for k, _ in flow.named_parameters()]
    for k in names:
        oracle.sd[k] = oracle.sd[k].clone().requires_grad_(True)
    gen = torch.Generator().manual_seed(12)
    R = orc.random_rotations(N, gen).to(dev)
    feat = torch.relu(torch.randn(N, F, generator=gen)).to(dev)
    opts = {"product": torch.optim.Adam(flow.parameters(), lr=1e-4),
            "oracle_eager": torch.optim.Adam([oracle.sd[k] for k in names], lr=1e-4)}
    losses = {k: [] for k in opts}

    def step(arm):
        if arm == "product":
            loss = -flow(R, feat)[1].mean()
        else:
            loss = -oracle.with_grad(R, feat)[1].mean()
        opts[arm].zero_grad(set_to_none=True)
        loss.backward()
        opts[arm].step()
        losses[arm].append(loss.detach())

    for _ in range(warmup):
        for arm in opts:
            step(arm)
    torch.cuda.synchronize()
    t = {k: [] for k in opts}
    for _ in range(reps):
        for arm in opts:
            t[arm].append(event_ms(lambda: step(arm)))
    prod, orac = statistics.median(t["product"]), statistics.median(t["oracle_eager"])
    return dict(config="modelnet_fisher", rot=rot, affine_layer=type(flow.layers[1]).__name__, F=F, layers=len(flow.layers), batch=N,
                product_ms_median=prod, oracle_eager_ms_median=orac, product_ms_all=t["product"], oracle_eager_ms_all=t["oracle_eager"],
                speedup_product_over_oracle_eager=orac / prod, product_rotations_per_s=N / (prod * 1e-3),
                loss_first_last={k: [float(v[0]), float(v[-1])] for k, v in losses.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--batches", default="4096,32768")
    ap.add_argument("--rots", default="36Trans,9TransLSmith")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "ablation_train_bench measures on the GPU"
    dev = torch.device("cuda", 0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        smi = "nvidia-smi not found"
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit_sm_clock_max_sm_clock=smi, warmup=args.warmup,
               reps=args.reps, timing="CUDA events around each full step (forward, backward, Adam), median; the arms alternate step by step",
               runs=[])
    for rot in args.rots.split(","):
        for N in (int(b) for b in args.batches.split(",")):
            r = run_config(rot, N, dev, args.warmup, args.reps)
            res["runs"].append(r)
            print(json.dumps({k: v for k, v in r.items() if not k.endswith("_all")}), flush=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
