"""Offline check of the inverse kernel's Newton stopping rule (csrc/flow_row.cu: stop on the predicted error of the next iterate)
on HARD synthetic mixtures: K = 64 components with |w'| up to 0.7 and peaky weights, evaluated in float32 like the kernel; the root
it stops at is compared with the float64 root.  What has to hold: |t_stop - t_true| * F' stays far inside the 2e-6 band in which
the replay of the reference's halvings evaluates explicitly instead of trusting sign(x0 - t*).
The "avg" rows start the iteration at the closed-form inverse of the Mobius map of the weighted mean centre.  The kernel starts
at pi: that start was measured on the device (DESIGN.md section 4.1) and removed; its code is in commit d73682a."""
import math
import numpy as np

rng = np.random.default_rng(0)
N, K = 20000, 64


def F64(t, a, b, pi, ys):
    zr, zv = np.cos(t)[:, None], np.sin(t)[:, None]
    dr, dv = zr - a, zv - b
    dd = dr * dr + dv * dv
    return t + 2 * (pi * np.arcsin((zr * dv - zv * dr) / np.sqrt(dd))).sum(1) - ys, (pi * (1 - a * a - b * b) / dd).sum(1)


def F32(t, a, b, pi, ys):
    f = np.float32
    zr, zv = np.cos(t).astype(f)[:, None], np.sin(t).astype(f)[:, None]
    dr, dv = zr - a, zv - b
    dd = dr * dr + dv * dv
    rs = (f(1) / np.sqrt(dd)).astype(f)
    m = ((zr * dv - zv * dr) * rs).astype(f)
    d = (pi * np.arcsin(m).astype(f)).sum(1, dtype=f)
    dF = (pi * (f(1) - a * a - b * b) * rs * rs).sum(1, dtype=f)
    return (t + f(2) * d - ys).astype(f), dF.astype(f)


for name, rad, peak in (("moderate", 0.4, 1.0), ("hard", 0.7, 3.0), ("extreme", 0.7, 6.0)):
    rho = rad * np.sqrt(rng.random((N, K))) if name != "extreme" else rad * (1 - 0.05 * rng.random((N, K)))
    ph = 2 * math.pi * rng.random((N, K))
    a, b = rho * np.cos(ph), rho * np.sin(ph)
    lg = peak * rng.standard_normal((N, K))
    pi = np.exp(lg - lg.max(1, keepdims=True)); pi /= pi.sum(1, keepdims=True)
    # the flow's own target: the moving column seen in its own frame sits at the angle pi (flow/mobiusflow.py:157-167)
    ys = np.full(N, math.pi)
    # float64 root by bisection
    lo, hi = np.full(N, math.pi / 2), np.full(N, 1.5 * math.pi)
    for _ in range(60):
        mid = 0.5 * (lo + hi)
        neg = F64(mid, a, b, pi, ys)[0] < 0
        lo, hi = np.where(neg, mid, lo), np.where(neg, hi, mid)
    root = 0.5 * (lo + hi)
    a32, b32, pi32, ys32 = (x.astype(np.float32) for x in (a, b, pi, ys))
    wb = (pi * a).sum(1) + 1j * (pi * b).sum(1)                    # weighted mean centre: ONE Mobius map, inverted in closed form
    z0 = (np.exp(1j * ys) + wb) / (1 + np.conj(wb) * np.exp(1j * ys))
    t_avg = np.clip(np.mod(np.angle(z0), 2 * math.pi), math.pi / 2 + 1e-3, 1.5 * math.pi - 1e-3).astype(np.float32)
    for predict, start in ((False, "pi"), (True, "pi"), (True, "avg")):
        ts = np.full(N, math.pi, np.float32) if start == "pi" else t_avg.copy()
        lo, hi = np.full(N, math.pi / 2, np.float32), np.full(N, 1.5 * math.pi, np.float32)
        conv = np.zeros(N, bool); prev = np.zeros(N, np.float32); ev = np.zeros(N, int); dFs = np.ones(N, np.float32)
        for it in range(10):
            Fv, dF = F32(ts, a32, b32, pi32, ys32)
            act = ~conv
            ev[act] += 1
            lo = np.where(act & (Fv < 0), ts, lo); hi = np.where(act & (Fv >= 0), ts, hi)
            dFs = np.where(act, dF, dFs)
            step = (Fv / dF).astype(np.float32); as_ = np.abs(step)
            c = as_ < 1e-5
            if predict:
                with np.errstate(divide="ignore", invalid="ignore"):
                    C = np.maximum(as_ / (prev * prev), np.float32(2))
                c = c | ((prev > 0) & (as_ < 1e-2) & (C * as_ * as_ < 5e-8))
            tn = (ts - step).astype(np.float32)
            bad = ~c & ~((tn > lo) & (tn < hi))
            pn = np.where(bad, np.float32(0), as_)
            tn = np.where(bad, (np.float32(0.5) * (lo + hi)).astype(np.float32), tn)
            ts = np.where(act, tn, ts); prev = np.where(act, pn, prev)
            conv = conv | (act & c)
            if conv.all():
                break
        err = np.abs(ts.astype(np.float64) - root) * dFs
        warp = ev.reshape(-1, 32).max(1)
        print(f"{name:9s} predict={int(predict)} start={start:3s}: converged {conv.mean():.4f}  evaluations per row {ev.mean():.2f} (warp max {warp.mean():.2f})  "
              f"|t - t*| F': median {np.median(err):.1e}  99.9% {np.quantile(err, 0.999):.1e}  max {err[conv].max():.1e}  (band 2e-6)")
