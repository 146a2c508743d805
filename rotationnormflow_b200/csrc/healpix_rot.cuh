// healpix_rot.cuh -- HEALPix SO(3) grid index -> fp32 rotation, shared by healpix_grid_kernel (healpix.cu) and the children kernel
// (hgrid.cu), so that a child's rotation is bit for bit the grid's row at that index.
//
// Follows utils/sd.py:48-82 (generate_healpix_grid): nside = 2^level, pixel centres from healpy.pix2vec in RING order (public
// HEALPix definition, SURVEY.md A.7), azimuth = atan2(y, x), polar = acos(z), tilts = linspace(0, 2 pi, 6*nside, endpoint=False),
// R[t*npix + b] = Rx(az_b) Rz(polar_b) Rx(tilt_t), all in float64 and rounded to float32 at the end (torch.Tensor(Rs), utils/sd.py:82).
#pragma once
#include <stdint.h>

namespace rnf {

__device__ __forceinline__ long long isqrt_ll(long long v) {
  long long r = (long long)sqrt((double)v);
  while (r * r > v) --r;
  while ((r + 1) * (r + 1) <= v) ++r;
  return r;
}

__device__ __forceinline__ void pix2zphi_ring(long long nside, long long p, double& z, double& phi) {
  const long long npix = 12 * nside * nside;
  const long long ncap = 2 * nside * (nside - 1);
  const double halfpi = 1.5707963267948966;
  if (p < ncap) {  // north polar cap
    const long long i = (1 + isqrt_ll(1 + 2 * p)) >> 1;
    const long long j = p + 1 - 2 * i * (i - 1);
    z = 1.0 - (double)(i * i) * (4.0 / (double)npix);
    phi = ((double)j - 0.5) * halfpi / (double)i;
  } else if (p < npix - ncap) {  // equatorial belt
    const long long ip = p - ncap;
    const long long i = ip / (4 * nside) + nside;
    const long long j = ip % (4 * nside) + 1;
    const double fodd = ((i + nside) & 1) ? 1.0 : 0.5;
    z = (double)(2 * nside - i) * (2.0 / (double)(3 * nside));
    phi = ((double)j - fodd) * halfpi / (double)nside;
  } else {  // south polar cap
    const long long ip = npix - p;
    const long long i = (1 + isqrt_ll(2 * ip - 1)) >> 1;
    const long long j = 4 * i + 1 - (ip - 2 * i * (i - 1));
    z = -1.0 + (double)(i * i) * (4.0 / (double)npix);
    phi = ((double)j - 0.5) * halfpi / (double)i;
  }
}

// rotation of grid index idx = t * npix + b at `level` (0 <= idx < 72 * 8^level), row-major fp32
__device__ __forceinline__ void healpix_rotation(int level, long long idx, float* o) {
  const long long nside = 1LL << level;
  const long long npix = 12 * nside * nside;
  const long long ntilt = 6 * nside;
  const long long t = idx / npix, b = idx % npix;
  double z, phi;
  pix2zphi_ring(nside, b, z, phi);
  const double sth = sqrt((1.0 - z) * (1.0 + z));
  const double az = atan2(sth * sin(phi), sth * cos(phi));
  const double polar = acos(z);
  const double tilt = (double)t * (6.283185307179586 / (double)ntilt);
  double sa, ca, sp, cp, st, ct;
  sincos(az, &sa, &ca);
  sincos(polar, &sp, &cp);
  sincos(tilt, &st, &ct);
  // Rx(az) Rz(polar), then times Rx(tilt)
  const double m00 = cp, m01 = -sp, m10 = ca * sp, m11 = ca * cp, m12 = -sa, m20 = sa * sp, m21 = sa * cp, m22 = ca;
  o[0] = (float)m00;
  o[1] = (float)(m01 * ct);
  o[2] = (float)(-m01 * st);
  o[3] = (float)m10;
  o[4] = (float)(m11 * ct + m12 * st);
  o[5] = (float)(-m11 * st + m12 * ct);
  o[6] = (float)m20;
  o[7] = (float)(m21 * ct + m22 * st);
  o[8] = (float)(-m21 * st + m22 * ct);
}

}  // namespace rnf
