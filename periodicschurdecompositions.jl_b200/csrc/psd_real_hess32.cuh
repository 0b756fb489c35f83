// Periodic Hessenberg-triangular reduction for small problems (n <= 32), no Schur vectors:
// ONE WARP PER PROBLEM, output in the packed layout consumed by rpqr_eig32_kernel.
//
// Same mathematics as phessenberg! (PeriodicSchurDecompositions.jl:229-247): for each column
// i, factors p..2 get a QR-type reflector (rows i..n-1) that is pushed into the right
// neighbour from the right, then H_1 gets the Hessenberg reflector (rows i+1..n-1) which is
// pushed into H_p.  Lane L owns row L / column L; the only cross-lane operation per
// reflector is one warp-wide sum of squares.  Reflectors are used un-normalised,
// H = I + g u u^T with g = -2/(u^T u) (see psd_real_eig32.cuh).
#pragma once
#include "psd_real_eig32.cuh"

namespace psd {

struct Hess32Params {
  int n, p;
  long long batch;
  int left;             // :L orientation: internal factor j <- user factor p+1-j (:127-131)
  int ld;               // smem leading dimension (odd)
  const double* A;      // [batch][p][n*n]
  double* packed_out;   // [batch][pk_problem_stride(n,p)]
  unsigned long long* counter;
};

// One reflector step: generate from Aj[r0.., col]; apply from the left to Aj[r0.., col+1..],
// from the right to Am[:, r0..].  0-based.  All 32 lanes must call.
PSD_DEV void hess32_step(double* Aj, double* Am, int n, int ld, int r0, int col, int lane) {
  double* xc = Aj + col * ld;  // source column
  const double alpha = xc[r0];
  const double xr = (lane > r0 && lane < n) ? xc[lane] : 0.0;
  double ssq = warp_sum(xr * xr);
  if (ssq == 0.0) {
    // either an exactly zero tail (H = I, householder.jl:76-78) or underflow of the squares
    const double amax = warp_max(fabs(xr));
    if (amax == 0.0) return;
  }
  double nn = fma(alpha, alpha, ssq);
  double sc = 1.0;
  if (!(ssq > 1e-280 && nn < 1e280)) {
    // rare: rescale by an exact power of two so that the squares are representable
    const double m = fmax(warp_max(fabs(xr)), fabs(alpha));
    sc = pow2_rescale(m);
    const double y = xr * sc;
    ssq = warp_sum(y * y);
    nn = fma(alpha * sc, alpha * sc, ssq);
  }
  const double al = alpha * sc;
  const double nrm = nn * fast_rsqrt(nn);
  const double betas = -copysign(nrm, al);
  const double u0s = al - betas;
  // H = I + g u u^T with u = (u0s, sc*x[r0+1..]) ; fold sc into the coefficients
  const double gs = -2.0 * fast_rcp(fma(u0s, u0s, ssq));
  double g = gs, u0 = u0s, beta = betas;
  if (sc != 1.0) {  // for u = (u0, x) with u0 = u0s/sc
    g = gs * sc * sc;
    u0 = u0s / sc;
    beta = betas / sc;
  }
  if (Am != Aj) {
    // Left update of Aj (lane = column, columns col+1..n-1) and right update of Am (lane = row)
    // touch different matrices: both dot products and both updates run in the same loops, so the
    // two dependent chains overlap (instruction-level parallelism within the warp).
    const bool la = (lane > col && lane < n), rw = (lane < n);
    double* cl = Aj + (la ? lane : col + 1 < n ? col + 1 : col) * ld;  // inactive lanes read a valid column
    double* ar = Am + (rw ? lane : 0);
    double dl0 = u0 * cl[r0], dl1 = 0.0, dr0 = ar[r0 * ld] * u0, dr1 = 0.0;
#pragma unroll 2
    for (int k = r0 + 1; k < n; k += 2) {
      const bool p1 = k + 1 < n;
      const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0;
      const double l0 = cl[k], l1 = p1 ? cl[k + 1] : 0.0;
      const double q0 = ar[k * ld], q1 = p1 ? ar[(k + 1) * ld] : 0.0;
      dl0 = fma(x0, l0, dl0); dl1 = fma(x1, l1, dl1);
      dr0 = fma(q0, x0, dr0); dr1 = fma(q1, x1, dr1);
    }
    const double sl = g * (dl0 + dl1), sr = g * (dr0 + dr1);
    if (la) cl[r0] = fma(sl, u0, cl[r0]);
    if (rw) ar[r0 * ld] = fma(sr, u0, ar[r0 * ld]);
#pragma unroll 2
    for (int k = r0 + 1; k < n; k += 2) {
      const bool p1 = k + 1 < n;
      const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0;
      const double l0 = cl[k], l1 = p1 ? cl[k + 1] : 0.0;
      const double q0 = ar[k * ld], q1 = p1 ? ar[(k + 1) * ld] : 0.0;
      if (la) {
        cl[k] = fma(sl, x0, l0);
        if (p1) cl[k + 1] = fma(sl, x1, l1);
      }
      if (rw) {
        ar[k * ld] = fma(sr, x0, q0);
        if (p1) ar[(k + 1) * ld] = fma(sr, x1, q1);
      }
    }
    __syncwarp();
    if (lane == r0) xc[lane] = beta;
    else if (lane > r0 && lane < n) xc[lane] = 0.0;
    __syncwarp();
    return;
  }
  // left: columns col+1..n-1 of Aj (lane = column).  Loops are unrolled by 4 with independent
  // accumulators and predicated loads so that the shared-memory loads pipeline.
  if (lane > col && lane < n) {
    double* a = Aj + lane * ld;
    double d0 = u0 * a[r0], d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll 2
    for (int k = r0 + 1; k < n; k += 4) {
      const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
      const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
      const double a0 = a[k], a1 = p1 ? a[k + 1] : 0.0, a2 = p2 ? a[k + 2] : 0.0, a3 = p3 ? a[k + 3] : 0.0;
      d0 = fma(x0, a0, d0); d1 = fma(x1, a1, d1); d2 = fma(x2, a2, d2); d3 = fma(x3, a3, d3);
    }
    const double s = g * ((d0 + d1) + (d2 + d3));
    a[r0] = fma(s, u0, a[r0]);
#pragma unroll 2
    for (int k = r0 + 1; k < n; k += 4) {
      const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
      const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
      const double a0 = a[k], a1 = p1 ? a[k + 1] : 0.0, a2 = p2 ? a[k + 2] : 0.0, a3 = p3 ? a[k + 3] : 0.0;
      a[k] = fma(s, x0, a0);
      if (p1) a[k + 1] = fma(s, x1, a1);
      if (p2) a[k + 2] = fma(s, x2, a2);
      if (p3) a[k + 3] = fma(s, x3, a3);
    }
  }
  if (Am == Aj) __syncwarp();
  // right: rows 0..n-1 of Am (lane = row), columns r0..n-1
  if (lane < n) {
    double* a = Am + lane;
    double d0 = a[r0 * ld] * u0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll 2
    for (int k = r0 + 1; k < n; k += 4) {
      const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
      const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
      const double a0 = a[k * ld], a1 = p1 ? a[(k + 1) * ld] : 0.0, a2 = p2 ? a[(k + 2) * ld] : 0.0,
                   a3 = p3 ? a[(k + 3) * ld] : 0.0;
      d0 = fma(a0, x0, d0); d1 = fma(a1, x1, d1); d2 = fma(a2, x2, d2); d3 = fma(a3, x3, d3);
    }
    const double s = g * ((d0 + d1) + (d2 + d3));
    a[r0 * ld] = fma(s, u0, a[r0 * ld]);
#pragma unroll 2
    for (int k = r0 + 1; k < n; k += 4) {
      const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
      const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
      const double a0 = a[k * ld], a1 = p1 ? a[(k + 1) * ld] : 0.0, a2 = p2 ? a[(k + 2) * ld] : 0.0,
                   a3 = p3 ? a[(k + 3) * ld] : 0.0;
      a[k * ld] = fma(s, x0, a0);
      if (p1) a[(k + 1) * ld] = fma(s, x1, a1);
      if (p2) a[(k + 2) * ld] = fma(s, x2, a2);
      if (p3) a[(k + 3) * ld] = fma(s, x3, a3);
    }
  }
  __syncwarp();
  if (lane == r0) xc[lane] = beta;
  else if (lane > r0 && lane < n) xc[lane] = 0.0;
  __syncwarp();
}

extern __shared__ __align__(16) double psd_smem_hess[];

template <int NN, int PP>
__global__ void __launch_bounds__(256) rphess_warp32_kernel_t(Hess32Params P) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = NN ? NN : P.n, p = PP ? PP : P.p, ld = NN ? (NN % 2 == 0 ? NN + 1 : NN) : P.ld;
  const size_t nn = (size_t)n * n;
  const int fs = ld * n;  // doubles per staged factor
  double* S = psd_smem_hess + (size_t)warp * p * fs;
  const int psize = pk_problem_size(n, p);
  for (;;) {
    long long b = 0;
    if (lane == 0) b = (long long)atomicAdd(P.counter, 1ULL);
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= P.batch) break;
    const double* Ab = P.A + (size_t)b * p * nn;
    // stage the whole problem with asynchronous 8-byte copies (LDGSTS): every load of the
    // problem is in flight before the first one is waited for
    for (int j = 0; j < p; j++) {
      const double* src = Ab + (size_t)(P.left ? (p - 1 - j) : j) * nn;
      double* dst = S + j * fs;
      if (lane < n)
        for (int c = 0; c < n; c++) {
          const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + c * ld + lane);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(src + c * n + lane));
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();
    // normalise every factor by an exact power of two (see pk_problem_stride)
    int escale = 0;
    for (int j = 0; j < p; j++) {
      double* dst = S + j * fs;
      double m = 0.0;
      if (lane < n)
        for (int c = 0; c < n; c++) m = fmax(m, fabs(dst[c * ld + lane]));
      m = warp_max(m);
      if (m > 0.0 && m <= DBL_MAX) {
        const int s = pow2_shift(m);
        if (s != 0) {
          const double sc = scalbn(1.0, s);
          if (lane < n)
            for (int c = 0; c < n; c++) dst[c * ld + lane] *= sc;
          escale -= s;
        }
      }
    }
    __syncwarp();
    for (int i = 0; i < n - 1; i++) {
      for (int j = p - 1; j >= 1; j--) hess32_step(S + j * fs, S + (j - 1) * fs, n, ld, i, i, lane);
      if (n - (i + 1) > 1) hess32_step(S, S + (p - 1) * fs, n, ld, i + 1, i, lane);
    }
    // packed output: H1 with 3 subdiagonals of storage, H2..Hp with 1 (zeros below structure)
    double* dstb = P.packed_out + (size_t)b * (psize + PK_STATE);
    if (lane == 0) dstb[psize] = (double)escale;
    for (int j = 0; j < p; j++) {
      const int kl = (j == 0) ? 3 : 1;
      const int keep = (j == 0) ? 1 : 0;
      double* dst = dstb + ((j == 0) ? 0 : pk_size(3, n) + (j - 1) * pk_size(1, n));
      const double* src = S + j * fs;
      for (int c = 0; c < n; c++) {
        const int off = pk_off(kl, c);
        if (lane <= c + kl && lane < n) dst[off + lane] = (lane <= c + keep) ? src[c * ld + lane] : 0.0;
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------
// Two warps per problem (p >= 2; the chain-ahead kernel below replaces it where that is faster, see
// launch_real_eig32).  Shared memory holds only three problems per SM, so the plain
// kernel runs three warps per SM and every problem pays the full latency of its serial chain of
// p (n-1) reflector steps.  Here the two independent halves of a step run on two warps (two
// schedulers): warp 0 of the pair applies the reflector to the factor itself from the left, warp 1
// pushes it into the neighbour factor from the right; both generate the reflector redundantly
// from the same shared-memory column (no exchange), and one 64-thread named barrier per step
// orders the neighbour's update before the next reflector is generated from it.
// ---------------------------------------------------------------------------------------------
PSD_DEV void pair_barrier(int id) { asm volatile("bar.sync %0, 64;" ::"r"(id) : "memory"); }

PSD_DEV void hess32_step_pair(double* Aj, double* Am, int n, int ld, int r0, int col, int lane, int role, int barid) {
  double* xc = Aj + col * ld;  // source column
  const double alpha = xc[r0];
  const double xr = (lane > r0 && lane < n) ? xc[lane] : 0.0;
  double ssq = warp_sum(xr * xr);
  if (ssq == 0.0) {
    const double amax = warp_max(fabs(xr));
    if (amax == 0.0) return;  // H = I for both warps (same data, same decision)
  }
  double nn = fma(alpha, alpha, ssq);
  double sc = 1.0;
  if (!(ssq > 1e-280 && nn < 1e280)) {
    const double m = fmax(warp_max(fabs(xr)), fabs(alpha));
    sc = pow2_rescale(m);
    const double y = xr * sc;
    ssq = warp_sum(y * y);
    nn = fma(alpha * sc, alpha * sc, ssq);
  }
  const double al = alpha * sc;
  const double nrm = nn * fast_rsqrt(nn);
  const double betas = -copysign(nrm, al);
  const double u0s = al - betas;
  const double gs = -2.0 * fast_rcp(fma(u0s, u0s, ssq));
  double g = gs, u0 = u0s, beta = betas;
  if (sc != 1.0) {
    g = gs * sc * sc;
    u0 = u0s / sc;
    beta = betas / sc;
  }
  if (role == 0) {
    // left: columns col+1..n-1 of Aj (lane = column)
    if (lane > col && lane < n) {
      double* a = Aj + lane * ld;
      double d0 = u0 * a[r0], d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll 2
      for (int k = r0 + 1; k < n; k += 4) {
        const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
        const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
        const double a0 = a[k], a1 = p1 ? a[k + 1] : 0.0, a2 = p2 ? a[k + 2] : 0.0, a3 = p3 ? a[k + 3] : 0.0;
        d0 = fma(x0, a0, d0); d1 = fma(x1, a1, d1); d2 = fma(x2, a2, d2); d3 = fma(x3, a3, d3);
      }
      const double s = g * ((d0 + d1) + (d2 + d3));
      a[r0] = fma(s, u0, a[r0]);
#pragma unroll 2
      for (int k = r0 + 1; k < n; k += 4) {
        const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
        const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
        const double a0 = a[k], a1 = p1 ? a[k + 1] : 0.0, a2 = p2 ? a[k + 2] : 0.0, a3 = p3 ? a[k + 3] : 0.0;
        a[k] = fma(s, x0, a0);
        if (p1) a[k + 1] = fma(s, x1, a1);
        if (p2) a[k + 2] = fma(s, x2, a2);
        if (p3) a[k + 3] = fma(s, x3, a3);
      }
    }
  } else {
    // right: rows 0..n-1 of Am (lane = row), columns r0..n-1
    if (lane < n) {
      double* a = Am + lane;
      double d0 = a[r0 * ld] * u0, d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll 2
      for (int k = r0 + 1; k < n; k += 4) {
        const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
        const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
        const double a0 = a[k * ld], a1 = p1 ? a[(k + 1) * ld] : 0.0, a2 = p2 ? a[(k + 2) * ld] : 0.0,
                     a3 = p3 ? a[(k + 3) * ld] : 0.0;
        d0 = fma(a0, x0, d0); d1 = fma(a1, x1, d1); d2 = fma(a2, x2, d2); d3 = fma(a3, x3, d3);
      }
      const double s = g * ((d0 + d1) + (d2 + d3));
      a[r0 * ld] = fma(s, u0, a[r0 * ld]);
#pragma unroll 2
      for (int k = r0 + 1; k < n; k += 4) {
        const bool p1 = k + 1 < n, p2 = k + 2 < n, p3 = k + 3 < n;
        const double x0 = xc[k], x1 = p1 ? xc[k + 1] : 0.0, x2 = p2 ? xc[k + 2] : 0.0, x3 = p3 ? xc[k + 3] : 0.0;
        const double a0 = a[k * ld], a1 = p1 ? a[(k + 1) * ld] : 0.0, a2 = p2 ? a[(k + 2) * ld] : 0.0,
                     a3 = p3 ? a[(k + 3) * ld] : 0.0;
        a[k * ld] = fma(s, x0, a0);
        if (p1) a[(k + 1) * ld] = fma(s, x1, a1);
        if (p2) a[(k + 2) * ld] = fma(s, x2, a2);
        if (p3) a[(k + 3) * ld] = fma(s, x3, a3);
      }
    }
  }
  pair_barrier(barid);  // the neighbour's update is complete; nobody reads the source column any more
  if (role == 0) {
    if (lane == r0) xc[lane] = beta;
    else if (lane > r0 && lane < n) xc[lane] = 0.0;
  }
}

template <int NN, int PP>
__global__ void __launch_bounds__(512) rphess_pair32_kernel_t(Hess32Params P) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int grp = warp >> 1, role = warp & 1, barid = 1 + grp;
  const int n = NN ? NN : P.n, p = PP ? PP : P.p, ld = NN ? (NN % 2 == 0 ? NN + 1 : NN) : P.ld;
  const size_t nn = (size_t)n * n;
  const int fs = ld * n;  // doubles per staged factor
  double* S = psd_smem_hess + (size_t)grp * p * fs;
  __shared__ long long s_b[8];
  __shared__ int s_e[8];
  const int psize = pk_problem_size(n, p);
  for (;;) {
    if (role == 0 && lane == 0) s_b[grp] = (long long)atomicAdd(P.counter, 1ULL);
    pair_barrier(barid);
    const long long b = s_b[grp];
    if (b >= P.batch) break;
    const double* Ab = P.A + (size_t)b * p * nn;
    // each warp of the pair stages, normalises and later packs every other factor
    int escale = 0;
    for (int j = role; j < p; j += 2) {
      const double* src = Ab + (size_t)(P.left ? (p - 1 - j) : j) * nn;
      double* dst = S + j * fs;
      if (lane < n)
        for (int c = 0; c < n; c++) {
          const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + c * ld + lane);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(src + c * n + lane));
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();
    for (int j = role; j < p; j += 2) {
      double* dst = S + j * fs;
      double m = 0.0;
      if (lane < n)
        for (int c = 0; c < n; c++) m = fmax(m, fabs(dst[c * ld + lane]));
      m = warp_max(m);
      if (m > 0.0 && m <= DBL_MAX) {
        const int s = pow2_shift(m);
        if (s != 0) {
          const double sc = scalbn(1.0, s);
          if (lane < n)
            for (int c = 0; c < n; c++) dst[c * ld + lane] *= sc;
          escale -= s;
        }
      }
    }
    if (role == 1 && lane == 0) s_e[grp] = escale;
    pair_barrier(barid);
    if (role == 0) escale += s_e[grp];
    for (int i = 0; i < n - 1; i++) {
      for (int j = p - 1; j >= 1; j--) hess32_step_pair(S + j * fs, S + (j - 1) * fs, n, ld, i, i, lane, role, barid);
      if (n - (i + 1) > 1) hess32_step_pair(S, S + (p - 1) * fs, n, ld, i + 1, i, lane, role, barid);
    }
    pair_barrier(barid);  // includes the last deferred column write of warp 0
    double* dstb = P.packed_out + (size_t)b * (psize + PK_STATE);
    if (role == 0 && lane == 0) dstb[psize] = (double)escale;
    for (int j = role; j < p; j += 2) {
      const int kl = (j == 0) ? 3 : 1;
      const int keep = (j == 0) ? 1 : 0;
      double* dst = dstb + ((j == 0) ? 0 : pk_size(3, n) + (j - 1) * pk_size(1, n));
      const double* src = S + j * fs;
      for (int c = 0; c < n; c++) {
        const int off = pk_off(kl, c);
        if (lane <= c + kl && lane < n) dst[off + lane] = (lane <= c + keep) ? src[c * ld + lane] : 0.0;
      }
    }
    // the barrier at the top of the loop keeps the next problem's staging behind this packing
  }
}

// ---------------------------------------------------------------------------------------------
// Reflector chain ahead of the trailing updates (p >= 7).  Shared memory holds only three problems
// per SM, so every problem pays the latency of its serial chain of p (n-1) reflector steps.  Only
// a small part of a step lies on that chain; here one CHAIN warp per problem runs it and two
// update warps (LEFT, RIGHT) apply the rest of every step, up to p-2 steps behind.
//
// Step s = (r0, col, j -> m) generates a reflector from rows r0..n-1 of column col of factor j,
// applies it from the left to columns col+1..n-1 of factor j and from the right to columns
// r0..n-1 of factor m.  The order is j = p-1..1 with r0 = col = i and m = j-1, then the H_1 step
// (j = 0, m = p-1, col = i, r0 = i+1), for i = 0..n-2.
//   chain warp: generates the reflector (u0, g, beta) exactly as hess32_step_pair does, computes
//     the right coefficient of every row, s_r = g * (row r of factor m, columns r0..) . u, with the
//     same accumulators and order, updates column r0 of factor m (the next step generates from
//     it), publishes (x[r0+1..n-1], s_r, u0, g) to a ring slot, then writes (beta, 0, ..) into the
//     source column.
//   left warp: for each published step, in order, the left update of factor j (columns
//     col+1..n-1; dot product and update per column, unchanged).
//   right warp: for each published step, in order, the rank-1 right update of factor m, columns
//     r0+1..n-1: a = fma(s_r, x_k, a).
//   The left update of step s+1 works on the factor that step s updated from the right (factor m
//   of step s is factor j of step s+1), so the left warp waits for the right warp's step s first.
//   The right warp never waits for the left warp: its step s+k writes factor j_s only for
//   k = p-1 (mod p), and the chain cannot publish that step before both update warps are done
//   with step s (below).
// Every matrix element gets the same fma sequence, in the same order, as with the two-warp kernel:
// the factors, and everything computed from them, are bitwise the same.
//
// Lag rule.  Chain step s = (i, j) reads column i of factor j and columns >= r0 of factor m.
// The updates that write these are
//   - the left update of factor m by the step of column i-1 that generated from factor m
//     ((i-1, j-1), or the H_1 step (i-1, 0) when m = 0): p-1 steps back;
//   - the right update into factor m by (i-1, j): p steps back;
//   - the left update of factor j by (i-1, j): p steps back (column i is one of its columns);
//   - the right update into factor j by the step just before s: columns > i only (column i is
//     updated by the chain).
// For the H_1 step (i, 0) (column i of factor 0, columns >= i+1 of factor p-1): the left update of
// factor p-1 by (i, p-1) is p-1 steps back, the left update of factor 0 and the right update into
// factor p-1 by (i-1, 0) are p steps back, and the right update into factor 0 by (i, 1) writes
// columns > i only.  So chain step s may start once the update warps have finished step s-(p-1): the
// chain runs at most L = p-2 steps ahead (none for p = 2).  The updates of the steps in between
// neither write what the chain reads nor read or write what it writes (column r0 of factor m,
// column col of factor j); they read only the ring and the elements they update.  The ring has
// L+1 slots (at most AHEAD_RING, a smaller lead is always safe): before step s writes its slot the
// chain waits until both update warps have released that slot's previous step, s-(L+1).  That wait is
// the lag rule.  Slots are handed over with mbarriers (release on arrive, acquire on wait).
// ---------------------------------------------------------------------------------------------
constexpr int AHEAD_RING = 8;   // ring slots per problem
constexpr int AHEAD_ENT = 68;   // doubles per ring entry: x[32], s_r[32], u0, g, H = I flag, pad
constexpr int AHEAD_CTL = 28;   // control words per problem: 3 x AHEAD_RING mbarriers, problem index, escale
constexpr int AHEAD_WARPS = 3;  // warps per problem: chain, left updates, right updates

__host__ __device__ inline size_t ahead_problem_doubles(int n, int p, int ld) {
  return (size_t)p * ld * n + AHEAD_RING * AHEAD_ENT + AHEAD_CTL;
}

PSD_DEV unsigned ahead_u32(const void* q) { return (unsigned)__cvta_generic_to_shared(q); }
PSD_DEV void ahead_mbar_init(unsigned long long* b, int cnt) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ahead_u32(b)), "r"(cnt) : "memory");
}
PSD_DEV void ahead_mbar_arrive(unsigned long long* b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(ahead_u32(b)) : "memory");
}
PSD_DEV void ahead_mbar_wait(unsigned long long* b, unsigned parity) {
  unsigned ok;
  do {
    asm volatile(
        "{\n.reg .pred q;\nmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\nselp.u32 %0, 1, 0, q;\n}\n"
        : "=r"(ok)
        : "r"(ahead_u32(b)), "r"(parity)
        : "memory");
  } while (!ok);
}
PSD_DEV void group_barrier(int id, int nthr) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthr) : "memory"); }

// Position of a step in the ring of its warp group: slot, mbarrier phase parity of this use of the
// slot, and whether the slot has been used before (steps continue across problems).
struct AheadPos {
  int slot = 0;
  unsigned phase = 0;
  bool used = false;
  PSD_DEV void advance(int slots) {
    if (++slot == slots) {
      slot = 0;
      phase ^= 1u;
      used = true;
    }
  }
};

// Dot product of u = (u0, x[r0+1..n-1]) with a row or column (elements a[k * st]), with the tail
// staged in registers first so that all its shared-memory loads are in flight together.  The sum
// is formed exactly as the loops of hess32_step_pair form it: d0 starts from the head product,
// then chunks of four terms go to four accumulators (zeros past the end of the last chunk), and
// the result is (d0 + d1) + (d2 + d3).  v[] and x[] keep the loaded values for the update.
PSD_DEV double ahead_tail_dot(const double* a, int st, const double* xc, int r0, int len, double d0, double (&v)[32],
                              double (&x)[32]) {
#pragma unroll
  for (int t = 0; t < 32; t++) {
    const bool in = t < len;
    const int k = in ? r0 + 1 + t : r0;  // always a valid address, even if the load is speculated
    x[t] = in ? xc[k] : 0.0;
    v[t] = in ? a[k * st] : 0.0;
  }
  double d1 = 0.0, d2 = 0.0, d3 = 0.0;
#pragma unroll
  for (int c = 0; c < 8; c++) {
    if (4 * c < len) {
      d0 = fma(x[4 * c], v[4 * c], d0);
      d1 = fma(x[4 * c + 1], v[4 * c + 1], d1);
      d2 = fma(x[4 * c + 2], v[4 * c + 2], d2);
      d3 = fma(x[4 * c + 3], v[4 * c + 3], d3);
    }
  }
  return (d0 + d1) + (d2 + d3);
}

PSD_DEV void ahead_chain_step(double* Aj, double* Am, int n, int ld, int r0, int col, int lane, double* ring,
                              unsigned long long* full, unsigned long long* empty, const AheadPos& q) {
  double* ent = ring + q.slot * AHEAD_ENT;
  if (q.used) ahead_mbar_wait(empty + q.slot, q.phase ^ 1u);  // the lag rule (see above)
  double* xc = Aj + col * ld;  // source column
  const double alpha = xc[r0];
  const double xr = (lane > r0 && lane < n) ? xc[lane] : 0.0;
  double ssq = warp_sum(xr * xr);
  if (ssq == 0.0) {
    // either an exactly zero tail (H = I, householder.jl:76-78) or underflow of the squares
    const double amax = warp_max(fabs(xr));
    if (amax == 0.0) {  // H = I: an entry the update warps skip
      if (lane == 0) {
        ent[66] = 1.0;
        ahead_mbar_arrive(full + q.slot);
      }
      return;
    }
  }
  double nn = fma(alpha, alpha, ssq);
  double sc = 1.0;
  if (!(ssq > 1e-280 && nn < 1e280)) {
    // rare: rescale by an exact power of two so that the squares are representable
    const double m = fmax(warp_max(fabs(xr)), fabs(alpha));
    sc = pow2_rescale(m);
    const double y = xr * sc;
    ssq = warp_sum(y * y);
    nn = fma(alpha * sc, alpha * sc, ssq);
  }
  const double al = alpha * sc;
  const double nrm = nn * fast_rsqrt(nn);
  const double betas = -copysign(nrm, al);
  const double u0s = al - betas;
  // H = I + g u u^T with u = (u0s, sc*x[r0+1..]) ; fold sc into the coefficients
  const double gs = -2.0 * fast_rcp(fma(u0s, u0s, ssq));
  double g = gs, u0 = u0s, beta = betas;
  if (sc != 1.0) {  // for u = (u0, x) with u0 = u0s/sc
    g = gs * sc * sc;
    u0 = u0s / sc;
    beta = betas / sc;
  }
  // right coefficient of every row of Am (lane = row) from columns r0..n-1, then column r0
  if (lane < n) {
    double* a = Am + lane;
    double v[32], x[32];
    const double ar0 = a[r0 * ld];
    const double s = g * ahead_tail_dot(a, ld, xc, r0, n - r0 - 1, ar0 * u0, v, x);
    a[r0 * ld] = fma(s, u0, ar0);
    ent[32 + lane] = s;
  }
  if (lane > r0 && lane < n) ent[lane] = xr;  // the tail, before the column is overwritten
  if (lane == 0) {
    ent[64] = u0;
    ent[65] = g;
    ent[66] = 0.0;
  }
  __threadfence_block();
  __syncwarp();
  if (lane == 0) ahead_mbar_arrive(full + q.slot);
  if (lane == r0) xc[lane] = beta;
  else if (lane > r0 && lane < n) xc[lane] = 0.0;
  __syncwarp();
}

// Left warp, step s: wait until the right warp has finished step s-1 (the right update of the
// previous step wrote the columns of factor j this step reads), then release step s-1 (the chain
// may reuse its slot only after both update warps are done with it), then the left update.  The
// release of s-1 comes after the wait on the right warp, so the right warp cannot complete that
// slot's next use (s-1+slots) before the left warp has seen this one.
PSD_DEV void ahead_left_step(double* Aj, int n, int r0, int col, int ld, int lane, const double* ring,
                             unsigned long long* full, unsigned long long* empty, unsigned long long* mid,
                             const AheadPos& q, const AheadPos& prev, bool first) {
  if (!first) {
    ahead_mbar_wait(mid + prev.slot, prev.phase);
    if (lane == 0) ahead_mbar_arrive(empty + prev.slot);
  }
  const double* ent = ring + q.slot * AHEAD_ENT;
  ahead_mbar_wait(full + q.slot, q.phase);
  if (ent[66] != 0.0) return;  // H = I
  const double u0 = ent[64], g = ent[65];
  const double* xc = ent;  // x[r0+1..n-1] at the rows' own indices
  // columns col+1..n-1 of Aj (lane = column)
  if (lane > col && lane < n) {
    double* a = Aj + lane * ld;
    const int len = n - r0 - 1;
    double v[32], x[32];
    const double ar0 = a[r0];
    const double s = g * ahead_tail_dot(a, 1, xc, r0, len, u0 * ar0, v, x);
    a[r0] = fma(s, u0, ar0);
#pragma unroll
    for (int t = 0; t < 31; t++)
      if (t < len) a[r0 + 1 + t] = fma(s, x[t], v[t]);
  }
  __threadfence_block();
  __syncwarp();
}

// Right warp, step s: rank-1 update of columns r0+1..n-1 of Am (lane = row), then tell the left
// warp (mid) and the chain (empty).
PSD_DEV void ahead_right_step(double* Am, int n, int r0, int ld, int lane, const double* ring,
                              unsigned long long* full, unsigned long long* empty, unsigned long long* mid,
                              const AheadPos& q) {
  const double* ent = ring + q.slot * AHEAD_ENT;
  ahead_mbar_wait(full + q.slot, q.phase);
  if (ent[66] == 0.0 && lane < n) {
    const double s = ent[32 + lane];
    const double* xc = ent;
    double* a = Am + lane;
    const int len = n - r0 - 1;
    double v[32], x[32];
#pragma unroll
    for (int t = 0; t < 31; t++) {
      const bool in = t < len;
      const int k = in ? r0 + 1 + t : r0;
      x[t] = in ? xc[k] : 0.0;
      v[t] = in ? a[k * ld] : 0.0;
    }
#pragma unroll
    for (int t = 0; t < 31; t++)
      if (t < len) a[(r0 + 1 + t) * ld] = fma(s, x[t], v[t]);
  }
  __threadfence_block();
  __syncwarp();
  if (lane == 0) {
    ahead_mbar_arrive(mid + q.slot);
    ahead_mbar_arrive(empty + q.slot);
  }
}

template <int NN, int PP>
__global__ void __launch_bounds__(AHEAD_WARPS * 32 * 4) rphess_ahead32_kernel_t(Hess32Params P) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int gw = AHEAD_WARPS;  // chain, left, right
  const int grp = warp / gw, role = warp - grp * gw, barid = 1 + grp, nthr = gw * 32;
  const int n = NN ? NN : P.n, p = PP ? PP : P.p, ld = NN ? (NN % 2 == 0 ? NN + 1 : NN) : P.ld;
  const size_t nn = (size_t)n * n;
  const int fs = ld * n;  // doubles per staged factor
  double* S = psd_smem_hess + (size_t)grp * ahead_problem_doubles(n, p, ld);
  double* ring = S + (size_t)p * fs;
  unsigned long long* full = (unsigned long long*)(ring + AHEAD_RING * AHEAD_ENT);
  unsigned long long* empty = full + AHEAD_RING;
  unsigned long long* mid = empty + AHEAD_RING;
  long long* s_b = (long long*)(mid + AHEAD_RING);
  int* s_e = (int*)(s_b + 1);
  const int slots = (p - 1 < AHEAD_RING) ? p - 1 : AHEAD_RING;
  if (role == 0 && lane == 0)
    for (int k = 0; k < slots; k++) {
      ahead_mbar_init(full + k, 1);
      ahead_mbar_init(empty + k, 2);
      ahead_mbar_init(mid + k, 1);
    }
  __syncthreads();
  const int psize = pk_problem_size(n, p);
  AheadPos q;
  for (;;) {
    if (role == 0 && lane == 0) *s_b = (long long)atomicAdd(P.counter, 1ULL);
    group_barrier(barid, nthr);
    const long long b = *s_b;
    if (b >= P.batch) break;
    const double* Ab = P.A + (size_t)b * p * nn;
    // each warp of the group stages, normalises and later packs every gw-th factor
    int escale = 0;
    for (int j = role; j < p; j += gw) {
      const double* src = Ab + (size_t)(P.left ? (p - 1 - j) : j) * nn;
      double* dst = S + j * fs;
      if (lane < n)
        for (int c = 0; c < n; c++) {
          const unsigned sa = (unsigned)__cvta_generic_to_shared(dst + c * ld + lane);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(src + c * n + lane));
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncwarp();
    for (int j = role; j < p; j += gw) {
      double* dst = S + j * fs;
      double m = 0.0;
      if (lane < n)
        for (int c = 0; c < n; c++) m = fmax(m, fabs(dst[c * ld + lane]));
      m = warp_max(m);
      if (m > 0.0 && m <= DBL_MAX) {
        const int s = pow2_shift(m);
        if (s != 0) {
          const double sc = scalbn(1.0, s);
          if (lane < n)
            for (int c = 0; c < n; c++) dst[c * ld + lane] *= sc;
          escale -= s;
        }
      }
    }
    if (lane == 0) s_e[role] = escale;
    group_barrier(barid, nthr);
    if (role == 0) {
      for (int w = 1; w < gw; w++) escale += s_e[w];
      for (int i = 0; i < n - 1; i++) {
        for (int j = p - 1; j >= 1; j--) {
          ahead_chain_step(S + j * fs, S + (j - 1) * fs, n, ld, i, i, lane, ring, full, empty, q);
          q.advance(slots);
        }
        if (n - (i + 1) > 1) {
          ahead_chain_step(S, S + (p - 1) * fs, n, ld, i + 1, i, lane, ring, full, empty, q);
          q.advance(slots);
        }
      }
    } else if (role == 1) {
      AheadPos prev = q;
      bool first = true;
      for (int i = 0; i < n - 1; i++) {
        for (int j = p - 1; j >= 1; j--) {
          ahead_left_step(S + j * fs, n, i, i, ld, lane, ring, full, empty, mid, q, prev, first);
          prev = q;
          first = false;
          q.advance(slots);
        }
        if (n - (i + 1) > 1) {
          ahead_left_step(S, n, i + 1, i, ld, lane, ring, full, empty, mid, q, prev, first);
          prev = q;
          first = false;
          q.advance(slots);
        }
      }
      // release the last step of the problem once the right warp is done with it
      if (!first) {
        ahead_mbar_wait(mid + prev.slot, prev.phase);
        if (lane == 0) ahead_mbar_arrive(empty + prev.slot);
      }
    } else {
      for (int i = 0; i < n - 1; i++) {
        for (int j = p - 1; j >= 1; j--) {
          ahead_right_step(S + (j - 1) * fs, n, i, ld, lane, ring, full, empty, mid, q);
          q.advance(slots);
        }
        if (n - (i + 1) > 1) {
          ahead_right_step(S + (p - 1) * fs, n, i + 1, ld, lane, ring, full, empty, mid, q);
          q.advance(slots);
        }
      }
    }
    group_barrier(barid, nthr);  // every update and the chain's last column writes are complete
    double* dstb = P.packed_out + (size_t)b * (psize + PK_STATE);
    if (role == 0 && lane == 0) dstb[psize] = (double)escale;
    for (int j = role; j < p; j += gw) {
      const int kl = (j == 0) ? 3 : 1;
      const int keep = (j == 0) ? 1 : 0;
      double* dst = dstb + ((j == 0) ? 0 : pk_size(3, n) + (j - 1) * pk_size(1, n));
      const double* src = S + j * fs;
      for (int c = 0; c < n; c++) {
        const int off = pk_off(kl, c);
        if (lane <= c + kl && lane < n) dst[off + lane] = (lane <= c + keep) ? src[c * ld + lane] : 0.0;
      }
    }
    // the barrier at the top of the loop keeps the next problem's staging behind this packing
  }
}

}  // namespace psd
