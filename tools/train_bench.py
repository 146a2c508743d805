"""Timing of one training step (forward, backward, Adam; agent.py:49-87): Flow.log_prob in the fused kernels (csrc/flow_grad.cu)
against the per-layer operators of train.composed_run, alternated in one run.

    python tools/train_bench.py --out r04_train_bench.json

CUDA events around each step, median of --reps timed steps of each path after --warmup untimed ones; the two paths alternate step
by step.  Configurations (seeded weights, seeded inputs, one image per rotation as agent.py feeds them):
  symsol           settings/symsol.yml, F = 512, uniform base (the settings of bench.py's train_step)
  modelnet_fisher  settings/modelnet_fisher.yml, F = 2080, matrix-Fisher base with a per-image A
at batch 4096 and 32768.  The fused step is also broken into phases, each timed on its own: device packing (Mobius images, affine
blocks, per-image constants), the forward kernel, the backward kernel, the rest of loss.backward() (weight-gradient GEMMs, the
reductions and autograd through the packing), and the Adam step."""
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
from rotationnormflow_b200 import _cabi, engine, flow as flow_mod  # noqa: E402
from rotationnormflow_b200.fisher import fisher_constants  # noqa: E402
from oracle import rnf_oracle as orc  # noqa: E402


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def median_ms(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    return statistics.median(event_ms(fn) for _ in range(reps))


def build(name, dev):
    cfg = rnf.load_config(name)
    torch.manual_seed(0)
    np.random.seed(0)
    with contextlib.redirect_stdout(io.StringIO()):
        return rnf.get_flow(cfg).to(dev).train()


def run_config(name, fisher, N, dev, warmup, reps):
    flow = build(name, dev)
    F = flow.feature_dim
    gen = torch.Generator().manual_seed(12)
    R = orc.random_rotations(N, gen).to(dev)
    feat = torch.relu(torch.randn(N, F, generator=gen)).to(dev)
    idx = torch.arange(N, device=dev)
    A = (3.0 * torch.randn(N, 3, 3, generator=gen)).to(dev).requires_grad_(True) if fisher else None
    opt = torch.optim.Adam(list(flow.parameters()) + ([A] if fisher else []), lr=1e-4)
    losses = {"fused": [], "composed": []}

    def loss_fused():
        return -flow.log_prob(R, feat, feature_index=idx, fisher_A=A).mean()

    def loss_composed():
        Ro, lp = flow(R, feat)                             # autograd on: train.composed_run
        if fisher:
            A9, c = fisher_constants(A)
            lp = lp + (A9.reshape(-1, 3, 3) * Ro).sum(dim=(1, 2)) - c
        return -lp.mean()

    def step(path):
        loss = loss_fused() if path == "fused" else loss_composed()
        opt.zero_grad(set_to_none=True)
        loss.backward()
        opt.step()
        losses[path].append(loss.detach())

    for _ in range(warmup):
        step("fused")
        step("composed")
    torch.cuda.synchronize()
    t = {"fused": [], "composed": []}
    for _ in range(reps):
        for path in ("fused", "composed"):
            t[path].append(event_ms(lambda: step(path)))
    fused, composed = statistics.median(t["fused"]), statistics.median(t["composed"])

    # ---- phases of the fused step, each timed on its own --------------------------------------------------------------------------
    layers, perms = list(flow.layers), flow._perm_rows()
    tp = flow_mod._train_program(flow, layers, perms, F, R.device)
    idx32 = idx.to(torch.int32)

    def pack():
        tp.images()
        engine.condition_torch(layers, feat)

    with torch.no_grad():
        mob, aff = tp.images()
        cond = engine.condition_torch(layers, feat)
        weights = tp.weights(mob, aff)
    per_row = tp.n_mob * engine.TRAIN_RECORD_FLOATS + tp.n_aff * 16
    chunk = max(1, min(N, engine.TRAIN_WORKSPACE_BYTES // (4 * per_row)))
    ws = torch.empty((chunk * per_row,), device=dev)
    G_R = torch.empty((N, 3, 3), device=dev)
    g_ldj = torch.full((N,), -1.0 / N, device=dev)

    def bwd_kernel():
        for s in range(0, N, chunk):
            n = min(chunk, N - s)
            _cabi.launch("rnf_flow_train_backward", dev, tp.prog.handle, weights, R[s:s + n], n, cond, N, idx32[s:s + n], 0, None, g_ldj[s:s + n],
                         G_R[s:s + n], ws, int(ws.numel()))

    holder = {}

    def fwd_total():
        holder["loss"] = loss_fused()

    def bwd_total():
        opt.zero_grad(set_to_none=True)
        holder["loss"].backward()

    def backward_only():
        fwd_total()
        torch.cuda.synchronize()
        return event_ms(bwd_total)

    phases = {
        "device_packing": median_ms(pack, 2, reps),
        "forward_kernel": median_ms(lambda: tp.forward(weights, R, cond, N, idx32), 2, reps),
        "forward_total": median_ms(fwd_total, 2, reps),
        "backward_kernel": median_ms(bwd_kernel, 2, reps),
        "backward_total": statistics.median(backward_only() for _ in range(reps)),
        "adam": median_ms(opt.step, 2, reps),
    }
    phases["gemms_and_autograd_glue"] = phases["backward_total"] - phases["backward_kernel"]
    return dict(config=name, fisher=fisher, F=F, layers=len(layers), batch=N, chunk_rows=chunk,
                fused_ms_median=fused, composed_ms_median=composed, fused_ms_all=t["fused"], composed_ms_all=t["composed"],
                speedup_fused_over_composed=composed / fused, fused_rotations_per_s=N / (fused * 1e-3),
                composed_rotations_per_s=N / (composed * 1e-3),
                loss_first_last={k: [float(v[0]), float(v[-1])] for k, v in losses.items()}, fused_phases_ms=phases)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--batches", default="4096,32768")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "train_bench measures on the GPU"
    dev = torch.device("cuda", 0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True).stdout.strip()
    except OSError:
        smi = "nvidia-smi not found"
    res = dict(device=torch.cuda.get_device_name(0), nvidia_smi=smi, warmup=args.warmup, reps=args.reps,
               timing="CUDA events around each full step (forward, backward, Adam), median; fused and composed alternate step by step",
               runs=[])
    for name, fisher in (("symsol", False), ("modelnet_fisher", True)):
        for N in (int(b) for b in args.batches.split(",")):
            r = run_config(name, fisher, N, dev, args.warmup, args.reps)
            res["runs"].append(r)
            print(json.dumps({k: v for k, v in r.items() if not k.endswith("_all")}), flush=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
