// Real standard periodic Schur kernel: one CTA per periodic problem.
//
// Replaces, on device, the reference call chain
//   pschur!(A, lr)                    PeriodicSchurDecompositions.jl:120-152
//   phessenberg!(A) + Matrix(H.Q)     PeriodicSchurDecompositions.jl:213-259, 136-140
//   pschur!(H1, Hs; ...)              PeriodicSchurDecompositions.jl:322-1096
//   _gs2x2!                           rschur2x2.jl:9-96
// with the reference-default ALGO_CONFIG switches (:287-302): LAPACK-style shifts,
// LAPACK + Ahues-Tisseur convergence test with eps^(1+4/16), no early QR start, no extra RQ.
//
// Data layout: the p factors (and, when requested, the p Schur-vector matrices) of the
// problem live either in shared memory (leading dimension ldh, odd, so that both row-wise
// and column-wise warp accesses are bank-conflict free) or, when they do not fit, in place
// in global memory (L2 resident); the code below is written on generic pointers and is
// identical for both.  Factor index j is always the INTERNAL rightwards index: for the :L
// orientation internal j maps to user factor p+1-j (:127-131).
#pragma once
#include "psd_device.cuh"
#include "psd_real_qr.cuh"
#include "psd_real_eig32.cuh"

namespace psd {

struct RpschurParams {
  int n, p;
  long long batch;
  int left, wantT, wantZ, maxitfac;
  double* A;        // [batch][p][n*n]  in/out (user order)
  double* Z;        // [batch][p][n*n]  out (reference result order) or nullptr
  double* eig;      // [batch][n][2]
  int* info;        // [batch]
  int* iters;       // [batch] or nullptr: total QR iterations (reference `niter`)
  int use_smem;     // factors staged in shared memory?
  int ldh;          // leading dimension of staged matrices
  int reduce_only;  // 1: stop after the Hessenberg-triangular reduction (psd_rphess_batched)
  int skip_reduce;  // 1: input is already Hessenberg/triangular (pschur!(H1,Hs) entry, :322)
  int z_preset;     // with skip_reduce: Z already holds the Q_j of an earlier reduction (Q kwarg, :326)
  unsigned long long* counter;  // dynamic work queue over problems
  double* scratch;  // per-CTA small arrays when they do not fit in smem (or nullptr)
  long long scratch_stride;
  double* tau;         // reduce_only, not nullptr: LAPACK-packed output - the reflector vectors stay
                       // below the (sub)diagonal of A_j and tau[b][j-1][0..n-1] receives their scalars
                       // (Hessenberg(A[1], tau[1]), QR(A[j], tau[j]) of phessenberg!, :249-253)
  double* packed_out;  // reduce_only: write packed Hessenberg-triangular factors here instead
                       // of A ([batch][pk_problem_size(n,p)], layout of psd_real_eig32.cuh)
};

// ---------------------------------------------------------------------------------------
// Periodic Hessenberg-triangular reduction, PeriodicSchurDecompositions.jl:229-247, with
// the Schur-vector accumulation fused in: instead of storing LAPACK-packed reflectors and
// materialising Q afterwards (orghr/orgqr, :136-140) each reflector is applied to Z[j]
// from the right as it is generated (Q_j = H_1 H_2 ... H_{n-1}).
// Every warp recomputes the column norm redundantly so no broadcast step is needed; one CTA
// barrier per reflector.
// ---------------------------------------------------------------------------------------
// mode 0: left + right + Z, then finalise the column; mode 1: left only (no finalise);
// mode 2: right + Z only, then finalise.  Modes 1,2 serialise the two sides when the left
// and right targets are the same matrix (p == 1).
// tau_slot != nullptr: packed output - the scaled reflector vector (implicit leading 1) is kept
// below the pivot and tau is stored, instead of the exact zeros.
PSD_DEV void reduce_step(const RCtx& c, double* Aj, double* Ajm1, double* Zj, int r0, int col,
                         int mode = 0, double* tau_slot = nullptr) {
  const int n = c.n, ld = c.ldh;
  const int m = n - r0 + 1;  // reflector order
  if (m <= 1) return;
  const int lane = c.tid & 31;
  const double* x = &PSD_EL(Aj, ld, r0, col);
  const double alpha = x[0];
  double amax = 0.0;
  for (int k = 1 + lane; k < m; k += 32) amax = fmax(amax, fabs(x[k]));
  amax = warp_max(amax);
  if (amax == 0.0) {  // tau = 0, H = I  (householder.jl:76-78)
    __syncthreads();
    return;
  }
  double mm = fmax(amax, fabs(alpha));
  double s = 1.0;
  if (mm < 1e-140 || mm > 1e140) s = pow2_rescale(mm);
  double ssq = 0.0;
  for (int k = 1 + lane; k < m; k += 32) {
    double y = x[k] * s;
    ssq = fma(y, y, ssq);
  }
  ssq = warp_sum(ssq);
  const double al = alpha * s;
  const double beta = -copysign(sqrt(fma(al, al, ssq)), al);
  const double tau = (beta - al) / beta;
  const double tv = s / (al - beta);  // v_k = x_k * tv
  // H = I - tau w w^T, w = (1, tv*x[1:]).
  const int nL = (mode == 2) ? 0 : (n - col);  // columns col+1..n of Aj
  const int nR = (mode == 1) ? 0 : n;          // rows of A_{j-1}
  const int nZ = (Zj && mode != 1) ? n : 0;
  const int tot = nL + nR + nZ;
  for (int w = c.tid; w < tot; w += c.nt) {
    if (w < nL) {
      double* a = &PSD_EL(Aj, ld, r0, col + 1 + w);
      double d = 0.0;
      for (int k = 1; k < m; k++) d = fma(x[k], a[k], d);
      d = tau * fma(d, tv, a[0]);
      a[0] -= d;
      const double g = d * tv;
      for (int k = 1; k < m; k++) a[k] = fma(-g, x[k], a[k]);
    } else {
      double* a;
      int lda;
      if (w < nL + nR) {
        a = &PSD_EL(Ajm1, ld, 1 + (w - nL), r0);
        lda = ld;
      } else {
        a = &PSD_EL(Zj, c.ldz, 1 + (w - nL - nR), r0);
        lda = c.ldz;
      }
      double d = 0.0;
      for (int k = 1; k < m; k++) d = fma(a[(size_t)k * lda], x[k], d);
      d = tau * fma(d, tv, a[0]);
      a[0] -= d;
      const double g = d * tv;
      for (int k = 1; k < m; k++) a[(size_t)k * lda] = fma(-g, x[k], a[(size_t)k * lda]);
    }
  }
  __syncthreads();
  if (mode == 1) return;
  // column `col` of Aj below r0 is dead from here on: store beta and exact zeros (or the
  // reflector vector: every element is read and rewritten by the same thread).
  for (int k = c.tid; k < m; k += c.nt) {
    double* e = &PSD_EL(Aj, ld, r0 + k, col);
    *e = (k == 0) ? beta / s : (tau_slot ? *e * tv : 0.0);
  }
  if (tau_slot && c.tid == 0) *tau_slot = tau;
}

PSD_DEV void phessenberg_cta(const RCtx& c, bool wantZ, double* tau = nullptr) {
  const int n = c.n, p = c.p;
  if (wantZ) {
    for (int j = 1; j <= p; j++) {
      double* Zj = c.Zp(j);
      for (int e = c.tid; e < n * n; e += c.nt) {
        int r = e % n, cc = e / n;
        Zj[r + (size_t)cc * c.ldz] = (r == cc) ? 1.0 : 0.0;
      }
    }
  }
  __syncthreads();
  for (int i = 1; i <= n - 1; i++) {
    for (int j = p; j >= 2; j--)
      reduce_step(c, c.Hp(j), c.Hp(j - 1), wantZ ? c.Zp(j) : nullptr, i, i, 0, tau ? tau + (size_t)(j - 1) * n + (i - 1) : nullptr);
    double* t1 = tau ? tau + (i - 1) : nullptr;
    if (p > 1) {
      reduce_step(c, c.Hp(1), c.Hp(p), wantZ ? c.Zp(1) : nullptr, i + 1, i, 0, t1);
    } else {
      reduce_step(c, c.Hp(1), c.Hp(1), wantZ ? c.Zp(1) : nullptr, i + 1, i, 1);
      reduce_step(c, c.Hp(1), c.Hp(1), wantZ ? c.Zp(1) : nullptr, i + 1, i, 2, t1);
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------------------------------
// Kernel: persistent CTAs pull problems from a global counter (convergence-dependent run
// time per problem), stage the factors, reduce, iterate, and write results back.
// ---------------------------------------------------------------------------------------
extern __shared__ __align__(16) double psd_smem[];

__global__ void rpschur_kernel(RpschurParams P) {
  const int n = P.n, p = P.p, tid = threadIdx.x, nt = blockDim.x;
  const size_t nn = (size_t)n * n;
  __shared__ long long s_b;

  double* small = P.scratch ? (P.scratch + (long long)blockIdx.x * P.scratch_stride) : psd_smem;
  double* mats = P.scratch ? psd_smem : (psd_smem + rp_small_doubles(n, p));

  RCtx c;
  c.n = n; c.p = p; c.tid = tid; c.nt = nt;
  c.hdiag = small;
  c.hsub = c.hdiag + (n + 2);
  c.hsup = c.hsub + (n + 2);
  c.t0 = c.hsup + (n + 2);
  c.t1 = c.t0 + (n + 2);
  c.t2 = c.t1 + (n + 2);
  c.lre = c.t2 + (n + 2);
  c.lim = c.lre + (n + 2);
  c.hnorms = c.lim + (n + 2);

  const bool wantZ = P.wantZ && P.Z;
  const bool left = P.left != 0;

  for (;;) {
    if (tid == 0) s_b = (long long)atomicAdd(P.counter, 1ULL);
    __syncthreads();
    const long long b = s_b;
    __syncthreads();
    if (b >= P.batch) break;

    double* Ab = P.A + (size_t)b * p * nn;
    double* Zb = wantZ ? (P.Z + (size_t)b * p * nn) : nullptr;

    if (P.use_smem) {
      c.ldh = P.ldh; c.ldz = P.ldh;
      c.H = mats; c.hs = (long long)P.ldh * n;
      c.Z = mats + (size_t)p * P.ldh * n; c.zs = (long long)P.ldh * n;
      c.zmap_left = false;
      // stage: internal factor j <- user factor (left ? p+1-j : j)
      for (int j = 1; j <= p; j++) {
        const double* src = Ab + (size_t)((left ? (p + 1 - j) : j) - 1) * nn;
        double* dst = c.Hp(j);
        for (int e = tid; e < (int)nn; e += nt) {
          int r = e % n, cc = e / n;
          dst[r + (size_t)cc * c.ldh] = src[e];
        }
      }
    } else {
      c.ldh = n; c.ldz = n;
      if (left) {
        c.H = Ab + (size_t)(p - 1) * nn; c.hs = -(long long)nn;
      } else {
        c.H = Ab; c.hs = (long long)nn;
      }
      c.Z = Zb; c.zs = (long long)nn;
      c.zmap_left = left;
    }
    __syncthreads();

    if (!P.skip_reduce) {
      double* taub = P.tau ? P.tau + (size_t)b * p * n : nullptr;
      if (taub) {
        for (int e = tid; e < p * n; e += nt) taub[e] = 0.0;  // (tau = 0 where H = I)
        __syncthreads();
      }
      phessenberg_cta(c, wantZ, taub);
    } else {
      if (wantZ && !P.z_preset) {
        for (int j = 1; j <= p; j++) {
          double* Zj = c.Zp(j);
          for (int e = tid; e < (int)nn; e += nt) {
            int r = e % n, cc = e / n;
            Zj[r + (size_t)cc * c.ldz] = (r == cc) ? 1.0 : 0.0;
          }
        }
      } else if (wantZ && P.use_smem) {
        // preset Q_j of the caller (rightwards order only): stage them next to the factors
        for (int j = 1; j <= p; j++) {
          const double* src = Zb + (size_t)(j - 1) * nn;
          double* Zj = c.Zp(j);
          for (int e = tid; e < (int)nn; e += nt) {
            int r = e % n, cc = e / n;
            Zj[r + (size_t)cc * c.ldz] = src[e];
          }
        }
      }
      // enforce structure: :380-387, :406
      for (int j = 1; j <= p; j++) {
        double* Hj = c.Hp(j);
        const int keep = (j == 1) ? 1 : 0;
        for (int e = tid; e < (int)nn; e += nt) {
          int r = e % n, cc = e / n;
          if (r > cc + keep) Hj[r + (size_t)cc * c.ldh] = 0.0;
        }
      }
      __syncthreads();
    }

    int info = 0, niter = 0;
    if (!P.reduce_only) info = periodic_qr_cta(c, P.wantT != 0, wantZ, P.maxitfac, &niter);

    // write back
    if (!P.reduce_only) {
      double* eg = P.eig + (size_t)b * 2 * n;
      for (int k = tid; k < n; k += nt) {
        eg[2 * k] = c.lre[k + 1];
        eg[2 * k + 1] = c.lim[k + 1];
      }
      if (tid == 0) {
        P.info[b] = info;
        if (P.iters) P.iters[b] = niter;
      }
    }
    if (P.packed_out) {
      // packed factors, each normalised by an exact power of two (see pk_problem_stride)
      double* dstb = P.packed_out + (size_t)b * pk_problem_stride(n, p);
      for (int j = 1 + tid; j <= p; j += nt) c.hnorms[j] = 0.0;
      __syncthreads();
      for (int j = 1; j <= p; j++) {
        const double* src = c.Hp(j);
        double m = 0.0;
        for (int e = tid; e < (int)nn; e += nt) m = fmax(m, fabs(src[(e % n) + (size_t)(e / n) * c.ldh]));
        m = warp_max(m);
        if ((tid & 31) == 0)
          atomicMax((unsigned long long*)&c.hnorms[j], (unsigned long long)__double_as_longlong(m));
      }
      __syncthreads();
      int escale = 0;
      for (int j = 1; j <= p; j++) {
        const int kl = (j == 1) ? 3 : 1;
        double* dst = dstb + ((j == 1) ? 0 : pk_size(3, n) + (j - 2) * pk_size(1, n));
        const double* src = c.Hp(j);
        const double m = c.hnorms[j];
        double sc = 1.0;
        if (m > 0.0 && m <= DBL_MAX) {
          const int s = pow2_shift(m);
          sc = scalbn(1.0, s);
          escale -= s;
        }
        for (int e = tid; e < (int)nn; e += nt) {
          int r = e % n, cc = e / n;
          if (r <= cc + kl) dst[pk_off(kl, cc) + r] = src[r + (size_t)cc * c.ldh] * sc;
        }
      }
      if (tid == 0) dstb[pk_problem_size(n, p)] = (double)escale;
    } else if (P.use_smem) {
      if (P.wantT || P.reduce_only) {
        for (int j = 1; j <= p; j++) {
          double* dst = Ab + (size_t)((left ? (p + 1 - j) : j) - 1) * nn;
          const double* src = c.Hp(j);
          for (int e = tid; e < (int)nn; e += nt) {
            int r = e % n, cc = e / n;
            dst[e] = src[r + (size_t)cc * c.ldh];
          }
        }
      }
      if (wantZ) {
        for (int j = 1; j <= p; j++) {
          int s = (left && j > 1) ? (p + 2 - j) : j;
          double* dst = Zb + (size_t)(s - 1) * nn;
          const double* src = c.Zp(j);
          for (int e = tid; e < (int)nn; e += nt) {
            int r = e % n, cc = e / n;
            dst[e] = src[r + (size_t)cc * c.ldz];
          }
        }
      }
    }
    __syncthreads();
  }
}

}  // namespace psd
