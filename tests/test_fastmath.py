"""CPU checks of the constants baked into csrc/mobius_fast.cuh and csrc/mobius_pair.cuh (fp32 emulation of the polynomial
evaluation)."""
import re
import os

import numpy as np

from conftest import ROOT


def _fma32(a, b, c):
    return (a.astype(np.float64) * b.astype(np.float64) + np.float64(c)).astype(np.float32)


def _function_body(header, name):
    """Source of the device function whose definition starts with `name` in csrc/<header>, up to its closing brace."""
    src = open(os.path.join(ROOT, "rotationnormflow_b200", "csrc", header)).read()
    start = src.index(name)
    return src[start:src.index("\n}\n", start)]


def test_softplus_series_branch_of_mixture_pairs():
    """e (1 - e/2) against log1p(e) below the 2^-7 switch-over: relative error <= e^2/3, absolute <= 2e-7."""
    e = np.linspace(0, 0.0078125, 1001)[1:]
    series = e * (1 - e / 2)
    assert (np.abs(series - np.log1p(e)) / np.log1p(e)).max() < 2.1e-5
    assert np.abs(series - np.log1p(e)).max() < 2e-7
    # constants in mixture_pairs are the series coefficients divided by ln 2
    body = _function_body("mobius_pair.cuh", "void mixture_pairs")
    m = re.search(r"small\[j\] = mul2\(e\[j\], fma2\(e\[j\], bc\((-?[0-9.]+)f\), bc\(([0-9.]+)f\)\)\)", body)
    assert abs(float(m.group(2)) - 1 / np.log(2)) < 1e-12 and abs(float(m.group(1)) + 0.5 / np.log(2)) < 1e-12


def test_packed_asin_degree6_accuracy():
    """mobius_pair.cuh takes the mixture angles as asin of a sine (no division): float32 Horner emulation of the degree-6
    polynomial read back from the header, against asin on [0, 1/sqrt 2]."""
    body = _function_body("mobius_pair.cuh", "f32x2 asin_unit2_s")
    co = [float(v) for v in re.findall(r"bc\((-?[0-9.e-]+)f\)", body)]          # highest power first
    assert len(co) == 7
    m = np.linspace(0, 0.70711, 1_000_001).astype(np.float32)
    s = (m.astype(np.float64) * m).astype(np.float32)
    p = np.full_like(s, np.float32(co[0]))
    for c in co[1:]:
        p = _fma32(p, s, np.float32(c))
    ps = (p.astype(np.float64) * s).astype(np.float32)
    res = (ps.astype(np.float64) * m + m).astype(np.float32)
    assert np.abs(res.astype(np.float64) - np.arcsin(m.astype(np.float64))).max() < 6e-8
    # unit vector: atan(min / max) == asin(min)
    t = np.linspace(0, np.pi / 4, 1001)
    assert np.abs(np.arctan(np.sin(t) / np.cos(t)) - np.arcsin(np.sin(t))).max() < 1e-15


def test_sincos_2pi_polynomial_accuracy():
    """Float32 emulation of sincos_2pi (mobius_fast.cuh) over [0, 2 pi] with the constants read back from the header."""
    body = _function_body("mobius_fast.cuh", "void sincos_2pi")
    num = r"(-?[0-9.]+(?:e-?[0-9]+)?)f"
    two_over_pi, magic = map(float, re.search(r"fmaf\(t, %s, %s\)" % (num, num), body).groups())
    hi = float(re.search(r"fmaf\(kf, %s, t\)" % num, body).group(1))
    lo = float(re.search(r"fmaf\(kf, %s, r\)" % num, body).group(1))
    s3, s2 = map(float, re.search(r"ps = fmaf\(%s, z, %s\)" % (num, num), body).groups())
    s1 = float(re.search(r"ps = fmaf\(ps, z, %s\)" % num, body).group(1))
    c3, c2 = map(float, re.search(r"pc = fmaf\(%s, z, %s\)" % (num, num), body).groups())
    c1 = float(re.search(r"pc = fmaf\(pc, z, %s\)" % num, body).group(1))
    assert magic == 12582912.0 and abs(two_over_pi - 2 / np.pi) < 1e-9 and abs(-hi - lo - np.pi / 2) < 1e-14
    f32 = lambda x: np.asarray(x).astype(np.float32)
    t = np.linspace(0, 2 * np.pi, 1_000_001).astype(np.float32)
    kf = f32(np.rint(t.astype(np.float64) * np.float32(two_over_pi)))
    r = f32(t.astype(np.float64) + kf.astype(np.float64) * np.float64(np.float32(hi)))
    r = f32(r.astype(np.float64) + kf.astype(np.float64) * np.float64(np.float32(lo)))
    z = f32(r * r)
    ps = f32(_fma32(f32(np.full_like(z, s3)), z, np.float32(s2)))
    ps = _fma32(ps, z, np.float32(s1))
    sn = f32(f32(ps * z).astype(np.float64) * r + r)
    pc = _fma32(f32(np.full_like(z, c3)), z, np.float32(c2))
    pc = _fma32(pc, z, np.float32(c1))
    cs = f32(f32(pc * z).astype(np.float64) * z + f32(np.float32(1) - np.float32(0.5) * z))
    q = kf.astype(np.int64) & 3
    S = np.where(q == 0, sn, np.where(q == 1, cs, np.where(q == 2, -sn, -cs)))
    C = np.where(q == 0, cs, np.where(q == 1, -sn, np.where(q == 2, -cs, sn)))
    assert np.abs(S - np.sin(t.astype(np.float64))).max() < 1.2e-7
    assert np.abs(C - np.cos(t.astype(np.float64))).max() < 1.2e-7


def test_half_angle_identity_of_the_forward_angle():
    """mixture_pairs (forward) takes theta = pi + 2 atan(q), q = -(tan of half the angle of h from the negative r axis) =
    -h_v / (1 - h_r) (= b' / Dn in the kernel's variables), |q| <= tan(asin 0.7), and evaluates atan(q) as asin(b' / |D|):
    the half-angle identity against atan2 wrapped to [0, 2 pi) over the left half plane."""
    qmax = np.tan(np.arcsin(0.7))
    psi = np.linspace(-2 * np.arcsin(0.7), 2 * np.arcsin(0.7), 100001)
    hr, hv = -np.cos(psi), np.sin(psi)                                   # unit vector within +-2 asin(0.7) of the angle pi
    ref = np.arctan2(hv, hr)
    ref = np.where(ref >= 0, ref, ref + 2 * np.pi)
    qq = -hv / (1 - hr)
    assert np.abs(qq).max() <= qmax * (1 + 1e-12)
    assert np.abs(np.pi + 2 * np.arctan(qq) - ref).max() < 1e-14


def test_scaled_forward_component_algebra():
    """The u-scaled forward evaluation of mixture_pairs (no reciprocal of u = 1 + |w|) against the textbook formulas
    (flow/mobiusflow.py:17-24,72,94-99), float64, random centres of any magnitude.  The half-angle step uses |h| = 1, i.e.
    a unit moving column; a column of norm 1 + eps moves the angle by O(eps), like the asin form it replaces."""
    rng = np.random.default_rng(0)
    n = 100000
    sc = 10 ** rng.uniform(-3, 2, n)
    a, b = rng.standard_normal(n) * sc, rng.standard_normal(n) * sc
    zr = -np.ones(n)
    nrm = np.sqrt(a * a + b * b)
    s = 0.7 / (1 + nrm)
    al, be = s * a, s * b
    dr, dv = zr - al, -be
    f = (1 - al * al - be * be) / (dr * dr + dv * dv)
    th = np.arctan2(f * dv - be, f * dr - al)
    th = np.where(th >= 0, th, th + 2 * np.pi)
    ap, bp = 0.7 * a, 0.7 * b
    rt = np.sqrt(ap * ap + bp * bp)
    u = 1 + rt / 0.7
    Dn = -zr * u + ap
    DD = Dn * Dn + bp * bp
    num = (rt * (1 / 0.49 - 1) + 2 / 0.7) * rt + 1
    f2 = num / DD
    q = bp / Dn                                                         # arg h = 2 arg(z - w') - arg z on the unit circle
    assert np.abs(q - (f2 * bp + bp) / (u + f2 * Dn + ap)).max() < 1e-12  # == -h_v / (1 - h_r), the half-angle tangent of h itself
    assert (np.abs(f2 - f) / f).max() < 1e-12
    assert np.abs(np.pi + 2 * np.arctan(q) - th).max() < 1e-12
    zr = -(1 + rng.uniform(-3e-7, 3e-7, n))                             # fp32-rounded column norm
    dr = zr - al
    f = (1 - al * al - be * be) / (dr * dr + dv * dv)
    th = np.arctan2(f * dv - be, f * dr - al)
    th = np.where(th >= 0, th, th + 2 * np.pi)
    Dn = -zr * u + ap
    f2 = num / (Dn * Dn + bp * bp)
    q = bp / Dn
    assert (np.abs(f2 - f) / f).max() < 1e-12 and np.abs(np.pi + 2 * np.arctan(q) - th).max() < 1e-6
