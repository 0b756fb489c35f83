// Device-side building blocks shared by the periodic Schur kernels (sm_100a).
//
// Execution model: one CTA owns one periodic problem.  Every thread of the CTA executes
// the same (convergence-dependent) control flow on values it reads from the problem's
// matrices after a CTA barrier, so scalar decisions (shifts, deflation, reflector
// generation for the 2- and 3-element bulge reflectors) are computed redundantly in
// registers by all threads with no broadcast step, while the row/column updates are
// spread over the threads (one row or one column per thread).
//
// Reference semantics restated here (file:line relative to the reference repository):
//   householder.jl:5-24     _norm2        -> power-of-two scaled sum of squares
//   householder.jl:66-108   _xreflector!  -> refl_small / refl_column
//   householder.jl:190-237  lmul!/rmul!   -> hh_apply<M>
//   householder.jl:269-304  HH2           -> hh_apply<2> with (v1,v2) whole vector
//   rschur2x2.jl:9-96       _gs2x2!       -> gs2x2
#pragma once
#include <cfloat>
#include <cstdint>
#include <cuda_runtime.h>

namespace psd {

#define PSD_DEV __device__ __forceinline__

// exponent s of the exact power-of-two scale 2^s that brings m > 0 into [0.5, 1), capped at 1000
// because 2^-e itself overflows for subnormal m.  A caller that records the scale of a factor must
// record this s, not -e: below 2^-1000 the two differ.
PSD_DEV int pow2_shift(double m) {
  int e;
  (void)frexp(m, &e);  // m = f * 2^e, f in [0.5,1)
  return (-e > 1000) ? 1000 : -e;
}

// exact power-of-two scale s = 2^-ilogb(m) for m > 0 (handles denormals)
PSD_DEV double pow2_rescale(double m) { return scalbn(1.0, pow2_shift(m)); }

// Reflector for a 2- or 3-vector held in registers.  On return x0 = beta, (v1,v2) the
// essential part, tau returned.  Same mathematics as householder.jl:66-108 (dlarfg); the
// overflow/underflow protection is an exact power-of-two prescale instead of the
// reference's scaled-ssq + sfmin loop, so results agree to rounding.
template <int M>
PSD_DEV double refl_small(double& x0, double& v1, double& v2) {
  double a1 = fabs(v1), a2 = (M == 3) ? fabs(v2) : 0.0;
  double amax = fmax(a1, a2);
  if (amax == 0.0) return 0.0;  // xnorm == 0: H = I, x untouched
  double m = fmax(amax, fabs(x0));
  double s = 1.0;
  if (m < 1e-140 || m > 1e140) s = pow2_rescale(m);
  double al = x0 * s, y1 = v1 * s, y2 = (M == 3) ? v2 * s : 0.0;
  double xn2 = y1 * y1 + y2 * y2;
  double beta = -copysign(sqrt(fma(al, al, xn2)), al);
  double tau = (beta - al) / beta;
  double t = 1.0 / (al - beta);
  v1 = y1 * t;
  if (M == 3) v2 = y2 * t;
  x0 = beta / s;
  return tau;
}

// Apply H = I - tau * w w^T, w = (1, v1[, v2]) to
//   L : from the left  to rows r..r+M-1, columns cl0..cl1   (one column per work item)
//   R : from the right to rows rr0..rr1, columns rc..rc+M-1 (one row per work item)
//   Zm: from the right to rows 1..nz,   columns zc..zc+M-1 (one row per work item)
// Work items are dealt round-robin to the nt threads.  1-based indices.
template <int M>
PSD_DEV void hh_apply(int tid, int nt, double* __restrict__ L, int ldl, int r, int cl0, int cl1,
                      double* __restrict__ R, int ldr, int rr0, int rr1, int rc,
                      double* __restrict__ Zm, int ldz, int nz, int zc, double v1, double v2,
                      double tau) {
  const int nL = (L && cl1 >= cl0) ? (cl1 - cl0 + 1) : 0;
  const int nR = (R && rr1 >= rr0) ? (rr1 - rr0 + 1) : 0;
  const int nZ = Zm ? nz : 0;
  const int tot = nL + nR + nZ;
  for (int w = tid; w < tot; w += nt) {
    if (w < nL) {
      double* a = L + (r - 1) + (size_t)(cl0 + w - 1) * ldl;
      double a0 = a[0], a1 = a[1], a2 = (M == 3) ? a[2] : 0.0;
      double s = a0 + v1 * a1;
      if (M == 3) s += v2 * a2;
      s *= tau;
      a[0] = a0 - s;
      a[1] = a1 - s * v1;
      if (M == 3) a[2] = a2 - s * v2;
    } else {
      double* a;
      int ld;
      if (w < nL + nR) {
        a = R + (rr0 + (w - nL) - 1) + (size_t)(rc - 1) * ldr;
        ld = ldr;
      } else {
        a = Zm + (w - nL - nR) + (size_t)(zc - 1) * ldz;
        ld = ldz;
      }
      double a0 = a[0], a1 = a[ld], a2 = (M == 3) ? a[2 * (size_t)ld] : 0.0;
      double s = a0 + a1 * v1;
      if (M == 3) s += a2 * v2;
      s *= tau;
      a[0] = a0 - s;
      a[ld] = a1 - s * v1;
      if (M == 3) a[2 * (size_t)ld] = a2 - s * v2;
    }
  }
}

// HH2 (householder.jl:269-304): whole 2-vector (w1,w2) stored, H = I - tau w w^T.
//   R : rows rr0..rr1, columns rc, rc+1 (right);  L : rows r, r+1, columns cl0..cl1 (left)
PSD_DEV void hh2_apply(int tid, int nt, double* __restrict__ L, int ldl, int r, int cl0, int cl1,
                       double* __restrict__ R, int ldr, int rr0, int rr1, int rc,
                       double* __restrict__ Zm, int ldz, int nz, int zc, double w1, double w2,
                       double tau) {
  const int nL = (L && cl1 >= cl0) ? (cl1 - cl0 + 1) : 0;
  const int nR = (R && rr1 >= rr0) ? (rr1 - rr0 + 1) : 0;
  const int nZ = Zm ? nz : 0;
  const int tot = nL + nR + nZ;
  const double t1 = w1 * tau, t2 = w2 * tau;
  for (int w = tid; w < tot; w += nt) {
    double *a, *b;
    if (w < nL) {
      a = L + (r - 1) + (size_t)(cl0 + w - 1) * ldl;
      b = a + 1;
    } else if (w < nL + nR) {
      a = R + (rr0 + (w - nL) - 1) + (size_t)(rc - 1) * ldr;
      b = a + ldr;
    } else {
      a = Zm + (w - nL - nR) + (size_t)(zc - 1) * ldz;
      b = a + ldz;
    }
    double a0 = *a, a1 = *b;
    double s = a0 * w1 + a1 * w2;
    *a = a0 - s * t1;
    *b = a1 - s * t2;
  }
}

// Plane rotation [c s; -s c]:
//   L : lmul!(G, .) on rows i1,i1+1, columns cl0..cl1
//   R : rmul!(., G') on rows rr0..rr1, columns rc, rc+1
//   Zm: rmul!(., G') on rows 1..nz, columns zc, zc+1
PSD_DEV void rot_apply(int tid, int nt, double* __restrict__ L, int ldl, int r, int cl0, int cl1,
                       double* __restrict__ R, int ldr, int rr0, int rr1, int rc,
                       double* __restrict__ Zm, int ldz, int nz, int zc, double c, double s) {
  const int nL = (L && cl1 >= cl0) ? (cl1 - cl0 + 1) : 0;
  const int nR = (R && rr1 >= rr0) ? (rr1 - rr0 + 1) : 0;
  const int nZ = Zm ? nz : 0;
  const int tot = nL + nR + nZ;
  for (int w = tid; w < tot; w += nt) {
    double *a, *b;
    if (w < nL) {
      a = L + (r - 1) + (size_t)(cl0 + w - 1) * ldl;
      b = a + 1;
    } else if (w < nL + nR) {
      a = R + (rr0 + (w - nL) - 1) + (size_t)(rc - 1) * ldr;
      b = a + ldr;
    } else {
      a = Zm + (w - nL - nR) + (size_t)(zc - 1) * ldz;
      b = a + ldz;
    }
    double a0 = *a, a1 = *b;
    *a = c * a0 + s * a1;
    *b = -s * a0 + c * a1;
  }
}

// LAPACK dlartg as transcribed by Julia's givensAlgorithm (real): [c s; -s c][f;g] = [r;0].
PSD_DEV void givens_real(double f, double g, double& cs, double& sn, double& r) {
  if (g == 0.0) {
    cs = 1.0; sn = 0.0; r = f;
  } else if (f == 0.0) {
    cs = 0.0; sn = 1.0; r = g;
  } else {
    double m = fmax(fabs(f), fabs(g));
    double s = 1.0;
    if (m < 1e-140 || m > 1e140) s = pow2_rescale(m);
    double f1 = f * s, g1 = g * s;
    double rr = sqrt(f1 * f1 + g1 * g1);
    cs = f1 / rr;
    sn = g1 / rr;
    r = rr / s;
    if (fabs(f) > fabs(g) && cs < 0.0) {
      cs = -cs; sn = -sn; r = -r;
    }
  }
}

// rschur2x2.jl:9-96 (_gs2x2! = LAPACK dlanv2).
PSD_DEV void gs2x2(double& a, double& b, double& c, double& d, double& cs, double& sn,
                   double& w1r, double& w1i, double& w2r, double& w2i) {
  const double half = 0.5, small = 4.0 * DBL_EPSILON;
#define PSD_SGN(x) (((x) < 0.0) ? -1.0 : 1.0)
  if (c == 0.0) {
    cs = 1.0; sn = 0.0;
  } else if (b == 0.0) {
    cs = 0.0; sn = 1.0;
    double ta = a;
    a = d; b = -c; c = 0.0; d = ta;
  } else if ((a - d) == 0.0 && (b * c < 0.0)) {
    cs = 1.0; sn = 0.0;
  } else {
    double asubd = a - d;
    double p = half * asubd;
    double bcmax = fmax(fabs(b), fabs(c));
    double bcmis = fmin(fabs(b), fabs(c)) * PSD_SGN(b) * PSD_SGN(c);
    double scale = fmax(fabs(p), bcmax);
    double z = (p / scale) * p + (bcmax / scale) * bcmis;
    if (z >= small) {
      z = p + sqrt(scale) * sqrt(z) * PSD_SGN(p);
      a = d + z;
      d -= (bcmax / z) * bcmis;
      double tau = hypot(c, z);
      cs = z / tau; sn = c / tau;
      b -= c; c = 0.0;
    } else {
      double sigma = b + c;
      double tau = hypot(sigma, asubd);
      cs = sqrt(half * (1.0 + fabs(sigma) / tau));
      sn = -(p / (tau * cs)) * PSD_SGN(sigma);
      double aa = a * cs + b * sn, bb = -a * sn + b * cs;
      double cc = c * cs + d * sn, dd = -c * sn + d * cs;
      a = aa * cs + cc * sn; b = bb * cs + dd * sn;
      c = -aa * sn + cc * cs; d = -bb * sn + dd * cs;
      double midad = half * (a + d);
      a = midad; d = a;
      if (c != 0.0) {
        if (b != 0.0) {
          if (b * c >= 0.0) {
            double sab = sqrt(fabs(b)), sac = sqrt(fabs(c));
            p = sab * sac * PSD_SGN(c);
            tau = 1.0 / sqrt(fabs(b + c));
            a = midad + p; d = midad - p;
            b -= c; c = 0.0;
            double cs1 = sab * tau, sn1 = sac * tau;
            double ncs = cs * cs1 - sn * sn1, nsn = cs * sn1 + sn * cs1;
            cs = ncs; sn = nsn;
          }
        } else {
          b = -c; c = 0.0;
          double t = cs;
          cs = -sn; sn = t;
        }
      }
    }
  }
#undef PSD_SGN
  if (c == 0.0) {
    w1r = a; w1i = 0.0; w2r = d; w2i = 0.0;
  } else {
    double rti = sqrt(fabs(b)) * sqrt(fabs(c));
    w1r = a; w1i = rti; w2r = d; w2i = -rti;
  }
}

PSD_DEV double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
PSD_DEV double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace psd
