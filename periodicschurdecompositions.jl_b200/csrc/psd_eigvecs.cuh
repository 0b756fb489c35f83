// Eigenvectors of a periodic Schur decomposition by periodic back-substitution: the analogue of
// LAPACK trevc for a product of triangular factors.  No eigenvalue is moved, so no periodic swap
// and no reordering is needed (the reference moves each eigenvalue to the top with ordschur!).
//
// Internal (rightwards) indexing, 0-based: factor R_j = T_j (:R) or T_{p-1-j} (:L), R_0 is the
// quasi-triangular Schur factor.  Vector x_j belongs to user vector u(j) = j (:R) or (p - j) mod p
// (:L), and v_u(j) = Z_u(j) x_j.  The relations are R_j x_{j+1} = mu_j x_j (x_p = x_0).
//
// For eigenvalue k fix x_j[k] = 1, so mu_j = R_j[k,k]; a complex pair's own 2x2 block takes x_0 as
// the eigenvector of the scaled 2x2 block product and x_j = B_j x_{j+1} normalised to x_j[k] = 1.
// Every row (or 2x2 row block) i above k then gives one cyclic system in x_0[i] .. x_{p-1}[i]:
//   -mu_j x_j[i] + R_j[i,i] x_{j+1}[i] = -s_j[i],   s_j[i] = sum_{i<m<=k} R_j[i,m] x_{j+1}[m],
// with determinant +-(prod R_j[i,i] - lambda_k), solved by a structured Givens QR (fill-in only
// in the last block column) after an exact power-of-two scaling of every row; a pivot below
// eps is replaced by eps as trevc does.  Each factor enters scaled by the power of two that brings
// its largest entry (in the leading part up to the problem's last vector) into [0.5, 1), which leaves every x_j
// unchanged, and each vector's chain x, s is rescaled by one common power of two whenever a solved
// row would take it near overflow.
//
// eigvecs_prep_kernel runs once per (problem, factor) first: the structure check and the factor
// exponents.  One CTA of eigvecs_kernel works on one problem and up to EV_CB eigenvectors ("slots"); warp q runs the cyclic
// solves of slot q, and the column-oriented s updates (s_j[r] += R_j[r,m] x_{j+1}[m], r < m) are
// spread over the CTA so that each column of T read serves every slot.  Small orders keep x and s
// in shared memory and finish in the kernel (back-transformation, normalisation, phase); large
// orders keep them in global memory and the host forms V_l = Z_l X_l with the DMMA GEMM before
// eigvecs_finish_kernel normalises.
#pragma once
#include "psd_gen_common.cuh"

namespace psd {

constexpr int EV_CB = 4;          // eigenvector slots per CTA
constexpr int EV_WS = 15;         // per slot and factor: mu + one block row of the QR (3*2*2 + 2)
constexpr int EV_LIM = 900;       // largest exponent a stored x may reach (s sums n terms of it)
constexpr double EV_BIG = 0x1p900;

struct EigvecParams {
  int n, p, left, nblk;       // nblk: CTAs per problem (grid.x = batch * nblk)
  long long batch;
  const void* T;              // [batch][p][n][n] storage layout, user factor order (double / cplx)
  const void* Z;
  const int* cols;            // [batch][n]: slot -> its (first) column, -1 past the last slot
  int32_t* info;              // [batch], zero on entry; 1 = not in periodic Schur form (prep kernel),
                              // 2 = a selected vector came out zero or non-finite
  int* fexp;                  // [batch][p]: exponent of the scale 2^-e of internal factor j (prep kernel)
  // shared-memory mode (global_mode == 0): V [batch][p][n][n] complex, zero on entry
  cplx* V;
  // global mode (one problem per launch): X [p][m][n] (user vector order), S [m][p][n], W [m][p][EV_WS]
  int global_mode, m;
  cplx* X;
  cplx* S;
  cplx* W;
};

PSD_DEV cplx ev_c(double v) { return mk(v, 0.0); }
PSD_DEV cplx ev_c(cplx v) { return v; }
// a = f 2^e, f in [0.5, 1) (frexp's e, read from the bit pattern: no library call); 0 for a zero
// or non-finite a
PSD_DEV int ev_exp(double a) {
  if (!(a > 0.0) || !isfinite(a)) return 0;
  const int ex = (int)((__double_as_longlong(a) >> 52) & 0x7ff);
  if (ex == 0) return (int)((__double_as_longlong(a * 0x1p64) >> 52) & 0x7ff) - 1022 - 64;  // subnormal
  return ex - 1022;
}

// Scaled product of the 2x2 diagonal blocks at rows i0, i0+1 of R_0 .. R_{p-1} (in that order),
// renormalised by a power of two after every factor (pow2_split): eigenvectors are unchanged.
template <class RF>
PSD_DEV void ev_block_product(int p, int i0, RF R, double (&P)[2][2]) {
  P[0][0] = 1.0; P[0][1] = 0.0; P[1][0] = 0.0; P[1][1] = 1.0;
  for (int j = 0; j < p; j++) {
    const double b00 = R(j, i0, i0), b01 = R(j, i0, i0 + 1), b10 = R(j, i0 + 1, i0), b11 = R(j, i0 + 1, i0 + 1);
    double Q[2][2];
    Q[0][0] = fma(P[0][0], b00, P[0][1] * b10);
    Q[0][1] = fma(P[0][0], b01, P[0][1] * b11);
    Q[1][0] = fma(P[1][0], b00, P[1][1] * b10);
    Q[1][1] = fma(P[1][0], b01, P[1][1] * b11);
    int e;
    (void)pow2_split(fmax(fmax(fabs(Q[0][0]), fabs(Q[0][1])), fmax(fabs(Q[1][0]), fabs(Q[1][1]))), e);
    for (int r = 0; r < 2; r++)
      for (int c = 0; c < 2; c++) P[r][c] = scalbn(Q[r][c], -e);
  }
}

// Discriminant of a 2x2 matrix: its eigenvalues are complex iff it is negative.
PSD_DEV double ev_disc(const double (&P)[2][2]) {
  const double h = 0.5 * (P[0][0] - P[1][1]);
  return fma(h, h, P[0][1] * P[1][0]);
}

// Cyclic block system of one row block (B = 1 or 2 rows) for one vector:
//   -mu_l u_l + D_l u_{l+1} = rhs_l  (l = 0..p-1, u_p = u_0),
// D(l, r, c) the scaled diagonal block of factor l, mu[l], rhs(l, r).  Structured Givens QR (the
// last block row is the spike; block row l keeps entries in block columns l, l+1 and p-1), rows
// scaled by exact powers of two first.  On return ws[l * (3 B^2 + B) + 3 B^2 + r] holds u_l[r] * 2^-E.
template <int B, class DF, class RF>
PSD_DEV void ev_cyclic_solve(int p, DF D, const cplx* mu, RF rhs, cplx* ws, int& E) {
  constexpr int RB = 3 * B * B + B;  // one stored block row: A (diag), Bm (next), F (last column), r
  const double smin = 2.220446049250313e-16;  // max(eps ||row||, smlnum) with rows scaled to ~1
  auto entry = [&](int l, int r, int cblk, int c) -> cplx {  // unscaled entry of block row l
    cplx v = mk(0.0, 0.0);
    if (cblk == l && r == c) v = -mu[l];
    if (cblk == (l + 1) % p) v = v + D(l, r, c);
    return v;
  };
  auto rowexp = [&](int l, int r) -> int {
    double mx = 0.0;
    for (int c = 0; c < B; c++) {
      mx = fmax(mx, amax_(entry(l, r, l, c)));
      if (p > 1) mx = fmax(mx, amax_(entry(l, r, (l + 1) % p, c)));
    }
    return ev_exp(mx);
  };
  // common exponent of the row-scaled right-hand sides
  int Er = -(1 << 30);
  for (int l = 0; l < p; l++)
    for (int r = 0; r < B; r++) {
      const cplx v = rhs(l, r);
      if (!is_zero(v)) Er = max(Er, ev_exp(amax_(v)) - rowexp(l, r));
    }
  if (Er == -(1 << 30)) Er = 0;
  auto load_row = [&](int l, int r, cplx (&Ad)[B][B], cplx (&Bn)[B][B], cplx& rr) {
    const int e = rowexp(l, r);
    for (int c = 0; c < B; c++) {
      Ad[r][c] = scal2(entry(l, r, l, c), -e);
      Bn[r][c] = (p > 1) ? scal2(entry(l, r, (l + 1) % p, c), -e) : mk(0.0, 0.0);
    }
    rr = scal2(rhs(l, r), -e - Er);
  };
  cplx G[B][B], S[B][B], rs[B];
  {
    cplx tmp[B][B];
    for (int r = 0; r < B; r++) load_row(p - 1, r, G, tmp, rs[r]);  // block column p-1 and block column 0
    for (int r = 0; r < B; r++)
      for (int c = 0; c < B; c++) S[r][c] = tmp[r][c];
  }
  for (int l = 0; l + 1 < p; l++) {
    cplx A[B][B], Bm[B][B], F[B][B], r[B], Sn[B][B];
    for (int rr = 0; rr < B; rr++) load_row(l, rr, A, Bm, r[rr]);
    const bool merge = (l + 2 == p);  // block column l+1 is the last one
    for (int rr = 0; rr < B; rr++)
      for (int c = 0; c < B; c++) {
        F[rr][c] = merge ? Bm[rr][c] : mk(0.0, 0.0);
        if (merge) Bm[rr][c] = mk(0.0, 0.0);
        Sn[rr][c] = mk(0.0, 0.0);
      }
    for (int cc = 0; cc < B; cc++)
      for (int ss = 0; ss < B; ss++) {
        if (is_zero(S[ss][cc])) continue;
        double c;
        cplx s, rv;
        givens_t(A[cc][cc], S[ss][cc], c, s, rv);
        auto rot = [&](cplx& t, cplx& b) {
          const cplx t2 = c * t + s * b;
          b = c * b - conj_(s) * t;
          t = t2;
        };
        for (int k = cc + 1; k < B; k++) rot(A[cc][k], S[ss][k]);
        for (int k = 0; k < B; k++) {
          rot(Bm[cc][k], Sn[ss][k]);
          rot(F[cc][k], G[ss][k]);
        }
        rot(r[cc], rs[ss]);
        A[cc][cc] = rv;
        S[ss][cc] = mk(0.0, 0.0);
      }
    cplx* w = ws + (size_t)l * RB;
    for (int rr = 0; rr < B; rr++) {
      for (int c = 0; c < B; c++) {
        w[rr * B + c] = A[rr][c];
        w[B * B + rr * B + c] = Bm[rr][c];
        w[2 * B * B + rr * B + c] = F[rr][c];
      }
      w[3 * B * B + rr] = r[rr];
    }
    for (int rr = 0; rr < B; rr++)
      for (int c = 0; c < B; c++) S[rr][c] = Sn[rr][c];
  }
  // last block row: G u_{p-1} = rs (a 2x2 G is triangularised by one more rotation)
  if (B == 2 && !is_zero(G[B - 1][0])) {
    double c;
    cplx s, rv;
    givens_t(G[0][0], G[B - 1][0], c, s, rv);
    const cplx g01 = c * G[0][B - 1] + s * G[B - 1][B - 1];
    G[B - 1][B - 1] = c * G[B - 1][B - 1] - conj_(s) * G[0][B - 1];
    G[0][B - 1] = g01;
    const cplx r0 = c * rs[0] + s * rs[B - 1];
    rs[B - 1] = c * rs[B - 1] - conj_(s) * rs[0];
    rs[0] = r0;
    G[0][0] = rv;
    G[B - 1][0] = mk(0.0, 0.0);
  }
  int se = 0;
  // back-substitution; a quotient that would pass EV_BIG rescales everything solved and unsolved
  auto solve_tri = [&](const cplx (&U)[B][B], cplx (&y)[B]) {
    for (int rr = B - 1; rr >= 0; rr--) {
      cplx num = y[rr];
      for (int c = rr + 1; c < B; c++) num = num - U[rr][c] * y[c];
      cplx pv = U[rr][rr];
      if (abs_(pv) < smin) pv = mk(smin, 0.0);
      const double an = amax_(num), ap = amax_(pv);
      if (an > EV_BIG * ap) {
        const int k = ev_exp(an) - ev_exp(ap) - EV_LIM + 2;
        for (int l = 0; l < p; l++)
          for (int c = 0; c < B; c++) ws[(size_t)l * RB + 3 * B * B + c] = scal2(ws[(size_t)l * RB + 3 * B * B + c], -k);
        for (int c = 0; c < B; c++) y[c] = scal2(y[c], -k);
        num = scal2(num, -k);
        se += k;
      }
      y[rr] = num / pv;
    }
  };
  {
    cplx* w = ws + (size_t)(p - 1) * RB;
    cplx y[B];
    for (int rr = 0; rr < B; rr++) {
      y[rr] = rs[rr];
      w[3 * B * B + rr] = rs[rr];
    }
    solve_tri(G, y);
    for (int rr = 0; rr < B; rr++) w[3 * B * B + rr] = y[rr];
  }
  for (int l = p - 2; l >= 0; l--) {
    cplx* w = ws + (size_t)l * RB;
    const cplx* un = ws + (size_t)(l + 1) * RB + 3 * B * B;
    const cplx* ul = ws + (size_t)(p - 1) * RB + 3 * B * B;
    cplx U[B][B], y[B];
    for (int rr = 0; rr < B; rr++) {
      cplx acc = w[3 * B * B + rr];
      for (int c = 0; c < B; c++) {
        U[rr][c] = w[rr * B + c];
        acc = acc - w[B * B + rr * B + c] * un[c] - w[2 * B * B + rr * B + c] * ul[c];
      }
      y[rr] = acc;
    }
    solve_tri(U, y);
    for (int rr = 0; rr < B; rr++) w[3 * B * B + rr] = y[rr];
  }
  E = Er + se;
}

// One column of V from its unnormalised values get(r), r < n, by one warp: unit 2-norm, the entry
// of largest modulus (lowest row on ties) real and positive; realvec zeroes the imaginary parts.
// out (and, when given, outc = its conjugate) are columns of V.  Returns false (and writes
// nothing) when the values are all zero or not finite.
template <class G>
PSD_DEV bool ev_finish_column(int n, int lane, G get, cplx* out, cplx* outc, bool realvec) {
  double am = -1.0;
  int im = n;
  for (int r = lane; r < n; r += 32) {
    const double a = abs_(get(r));
    if (a > am) { am = a; im = r; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    const double a2 = __shfl_xor_sync(0xffffffffu, am, o);
    const int i2 = __shfl_xor_sync(0xffffffffu, im, o);
    if (a2 > am || (a2 == am && i2 < im)) { am = a2; im = i2; }
  }
  if (!(am > 0.0) || !isfinite(am)) return false;  // V stays zero
  const int e = ev_exp(am);
  double ss = 0.0;
  for (int r = lane; r < n; r += 32) ss += sq_(scal2(get(r), -e));
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const double nrm = sqrt(ss);
  const cplx wm = scal2(get(im), -e);
  const double awm = abs_(wm);
  const cplx ph = conj_(wm) * (1.0 / (awm * nrm));
#pragma unroll 1
  for (int r = lane; r < n; r += 32) {
    cplx v = (r == im) ? mk(awm / nrm, 0.0) : scal2(get(r), -e) * ph;
    if (realvec) v.y = 0.0;
    out[r] = v;
    if (outc) outc[r] = conj_(v);
  }
  return true;
}

// Once per problem b = blockIdx.x and internal factor j = blockIdx.y, before eigvecs_kernel: the
// exponent e_j that brings the largest entry of the leading kk x kk part of R_j (kk - 1 = top row of
// the problem's last slot; the upper part and the first subdiagonal) into [0.5, 1), and, in the
// CTA of j = 0, the structure check (info = 1: two adjacent nonzero subdiagonal entries of R_0, a
// nonzero subdiagonal entry of another factor or of a complex R_0, or a 2x2 block of R_0 whose
// product has real eigenvalues).  Entries below the first subdiagonal are never read.
template <class T>
__global__ void __launch_bounds__(256) eigvecs_prep_kernel(EigvecParams P) {
  const int n = P.n, p = P.p, tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
  const long long b = blockIdx.x;
  const int j = blockIdx.y;
  const size_t nn = (size_t)n * n;
  const T* Tb = (const T*)P.T + (size_t)b * p * nn;
  const bool realT = sizeof(T) == sizeof(double);
  auto Rt = [&](int jj, int r, int c) -> T { return Tb[(size_t)(P.left ? p - 1 - jj : jj) * nn + r + (size_t)c * n]; };
  auto Rr = [&](int jj, int r, int c) -> double { return re_(Rt(jj, r, c)); };
  __shared__ int s_last, s_exp, s_bad;
  if (tid == 0) { s_last = -1; s_exp = -(1 << 30); s_bad = 0; }
  __syncthreads();
  for (int q = tid; q < n; q += nt)
    if (P.cols[(size_t)b * n + q] >= 0) atomicMax(&s_last, P.cols[(size_t)b * n + q]);
  if (j == 0)
    for (int r = 1 + tid; r < n; r += nt) {
      bool bad = false;
      if (!is_zero(Rt(0, r, r - 1))) {
        if (!realT || (r + 1 < n && !is_zero(Rt(0, r + 1, r)))) {
          bad = true;
        } else {
          double Pm[2][2];
          ev_block_product(p, r - 1, Rr, Pm);
          bad = !(ev_disc(Pm) < 0.0);
        }
      }
      for (int jj = 1; jj < p && !bad; jj++) bad = !is_zero(Rt(jj, r, r - 1));
      if (bad) s_bad = 1;
    }
  __syncthreads();
  if (j == 0 && tid == 0 && s_bad) P.info[b] = 1;
  const int c = s_last;
  const int kk = (c < 0) ? 0 : ((realT && c + 1 < n && !is_zero(Rt(0, c + 1, c))) ? c + 2 : c + 1);
  double mx = 0.0;
  for (int cc = tid >> 5; cc < kk; cc += nt >> 5)
#pragma unroll 1
    for (int r = lane; r <= min(cc + 1, kk - 1); r += 32) mx = fmax(mx, amax_(Rt(j, r, cc)));
  for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0 && mx > 0.0) atomicMax(&s_exp, ev_exp(mx));
  __syncthreads();
  if (tid == 0) P.fexp[(size_t)b * p + j] = (s_exp == -(1 << 30)) ? 0 : min(1000, max(-1000, s_exp));
}

template <class T>
__global__ void __launch_bounds__(256) eigvecs_kernel(EigvecParams P) {
  extern __shared__ __align__(16) double ev_smem[];
  const int n = P.n, p = P.p, tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const long long b = blockIdx.x / P.nblk;
  const int blk = blockIdx.x % P.nblk;
  const size_t nn = (size_t)n * n;
  const T* Tb = (const T*)P.T + (size_t)b * p * nn;
  const bool realT = sizeof(T) == sizeof(double);
  auto fac = [&](int j) { return P.left ? p - 1 - j : j; };
  auto uvec = [&](int j) { return P.left ? (p - j) % p : j; };
  auto Rt = [&](int j, int r, int c) -> T { return Tb[(size_t)fac(j) * nn + r + (size_t)c * n]; };
  auto Rr = [&](int j, int r, int c) -> double { return re_(Rt(j, r, c)); };  // real input only

  if (P.info[b] == 1) return;  // not in periodic Schur form (eigvecs_prep_kernel): V stays zero
  __shared__ int s_col[EV_CB], s_top[EV_CB];
  if (tid < EV_CB) {
    const int slot = blk * EV_CB + tid;
    const int c = (slot < n) ? P.cols[(size_t)b * n + slot] : -1;
    s_col[tid] = c;
    s_top[tid] = (c >= 0 && realT && c + 1 < n && !is_zero(Rt(0, c + 1, c))) ? c + 1 : c;
  }
  __syncthreads();
  int kmax = -1;
  for (int q = 0; q < EV_CB; q++) kmax = max(kmax, s_top[q]);
  if (kmax < 0) return;

  // ---- shared memory: factor scales, staging of the solved rows, [ws, x, s] ----
  const int p2 = (p + 1) & ~1;
  double* fsc = ev_smem;
  cplx* xst = (cplx*)(ev_smem + p2);               // [CB][p][2]: sc_j x_{j+1}[rows of the block]
  cplx* sm = xst + (size_t)EV_CB * p * 2;
  const size_t pn = (size_t)p * n;
  auto wsp = [&](int q) -> cplx* {
    return P.global_mode ? P.W + (size_t)(blk * EV_CB + q) * p * EV_WS : sm + (size_t)q * p * EV_WS;
  };
  auto xcol = [&](int q, int u) -> cplx* {  // x of user vector u
    return P.global_mode ? P.X + ((size_t)u * P.m + blk * EV_CB + q) * n
                         : sm + (size_t)EV_CB * p * EV_WS + ((size_t)q * p + u) * n;
  };
  auto scol = [&](int q, int j) -> cplx* {
    return P.global_mode ? P.S + ((size_t)(blk * EV_CB + q) * p + j) * n
                         : sm + (size_t)EV_CB * p * EV_WS + (size_t)EV_CB * pn + ((size_t)q * p + j) * n;
  };
  for (int j = tid; j < p; j += nt) fsc[j] = scalbn(1.0, -P.fexp[(size_t)b * p + j]);
  // ---- zero x and s of every live slot ----
  for (int q = 0; q < EV_CB; q++) {
    if (s_col[q] < 0) continue;
    for (size_t e = tid; e < pn; e += nt) {
      xcol(q, (int)(e / n))[e % n] = mk(0.0, 0.0);
      scol(q, (int)(e / n))[e % n] = mk(0.0, 0.0);
    }
  }
  __syncthreads();
  auto D = [&](int j, int r, int c, int i0) -> cplx { return ev_c(Rt(j, i0 + r, i0 + c)) * fsc[j]; };

  // ---- row blocks from kmax down ----
  for (int r = kmax; r >= 0;) {
    const bool two = realT && r >= 1 && !is_zero(Rt(0, r, r - 1));
    const int i0 = two ? r - 1 : r, bs = two ? 2 : 1;
    unsigned act = 0;
    for (int q = 0; q < EV_CB; q++)
      if (s_col[q] >= 0 && i0 <= s_col[q]) act |= 1u << q;
    if (warp < EV_CB && (act >> warp & 1u)) {
      const int q = warp;
      cplx* ws = wsp(q);
      cplx* mu = ws + (size_t)p * (EV_WS - 1);
      int E = 0, shift = 0;
      if (i0 == s_col[q]) {
        // the vector's own block: x_j[i0] = 1
        if (lane == 0) {
          if (bs == 1) {
            for (int j = 0; j < p; j++) {
              mu[j] = D(j, 0, 0, i0);
              ws[j * 2] = mk(1.0, 0.0);
            }
          } else {
            double Pm[2][2];
            ev_block_product(p, i0, Rr, Pm);
            const double t = 0.5 * (Pm[0][0] + Pm[1][1]);
            const cplx lam = mk(t, sqrt(fmax(0.0, -ev_disc(Pm))));
            cplx y1;  // x_0 = [1, y1]: eigenvector of the product for lam (Im lam > 0)
            const cplx lmd = lam - ev_c(Pm[1][1]);
            if (fabs(Pm[0][1]) >= abs_(lmd)) y1 = (lam - ev_c(Pm[0][0])) / Pm[0][1];
            else y1 = ev_c(Pm[1][0]) / lmd;
            // x_j = B_j x_{j+1} normalised to x_j[i0] = 1, j = p-1 .. 1; mu_j = (B_j x_{j+1})[i0]
            cplx nx = y1;  // second entry of x_{j+1}
            ws[0] = mk(1.0, 0.0);
            ws[1] = y1;
            for (int j = p - 1; j >= 0; j--) {
              const cplx z0 = D(j, 0, 0, i0) + D(j, 0, 1, i0) * nx;
              const cplx z1 = D(j, 1, 0, i0) + D(j, 1, 1, i0) * nx;
              mu[j] = z0;
              if (j > 0) {
                nx = z1 / z0;
                ws[j * 2] = mk(1.0, 0.0);
                ws[j * 2 + 1] = nx;
              }
            }
          }
        }
        __syncwarp();
        for (int j = lane; j < p; j += 32)
          for (int rr = 0; rr < bs; rr++) xcol(q, uvec(j))[i0 + rr] = ws[j * 2 + rr];
      } else {
        if (lane == 0) {
          auto rhs = [&](int l, int rr) -> cplx { return -scol(q, l)[i0 + rr]; };
          if (bs == 1) {
            auto Dj = [&](int j, int rr, int c) { return D(j, rr, c, i0); };
            ev_cyclic_solve<1>(p, Dj, mu, rhs, ws, E);
          } else {
            auto Dj = [&](int j, int rr, int c) { return D(j, rr, c, i0); };
            ev_cyclic_solve<2>(p, Dj, mu, rhs, ws, E);
          }
          const int RB = 3 * bs * bs + bs;
          int mx = -(1 << 30);
          for (int l = 0; l < p; l++)
            for (int rr = 0; rr < bs; rr++) {
              const cplx u = ws[(size_t)l * RB + 3 * bs * bs + rr];
              if (!is_zero(u)) mx = max(mx, ev_exp(amax_(u)));
            }
          if (mx != -(1 << 30) && E + mx > EV_LIM) shift = E + mx - EV_LIM;
        }
        E = __shfl_sync(0xffffffffu, E, 0);
        shift = __shfl_sync(0xffffffffu, shift, 0);
        __syncwarp();
        if (shift > 0) {  // common power of two on the whole chain x, s of this vector
          for (size_t e = lane; e < pn; e += 32) {
            cplx* xc = xcol(q, (int)(e / n));
            cplx* sc = scol(q, (int)(e / n));
            xc[e % n] = scal2(xc[e % n], -shift);
            sc[e % n] = scal2(sc[e % n], -shift);
          }
          E -= shift;
          __syncwarp();
        }
        const int RB = 3 * bs * bs + bs;
        for (int j = lane; j < p; j += 32)
          for (int rr = 0; rr < bs; rr++)
            xcol(q, uvec(j))[i0 + rr] = scal2(ws[(size_t)j * RB + 3 * bs * bs + rr], E);
      }
      __syncwarp();
      for (int j = lane; j < p; j += 32)
        for (int rr = 0; rr < bs; rr++)
          xst[((size_t)q * p + j) * 2 + rr] = xcol(q, uvec((j + 1) % p))[i0 + rr] * fsc[j];
    }
    __syncthreads();
    // s_j[r'] += R_j[r', m] sc_j x_{j+1}[m] for the rows r' < i0 of every live slot
    if (act && i0 > 0) {
      for (int e = tid; e < p * i0; e += nt) {
        const int j = e / i0, rr = e % i0;
        for (int c = 0; c < bs; c++) {
          const T t = Rt(j, rr, i0 + c);
#pragma unroll
          for (int q = 0; q < EV_CB; q++)
            if (act >> q & 1u) {
              cplx* sc = scol(q, j);
              sc[rr] = sc[rr] + t * xst[((size_t)q * p + j) * 2 + c];
            }
        }
      }
    }
    __syncthreads();
    r = i0 - 1;
  }
  if (P.global_mode) return;

  // ---- shared-memory mode: v_u = Z_u x (rows <= kmax of x are the only nonzero ones) ----
  const T* Zb = (const T*)P.Z + (size_t)b * p * nn;
  for (size_t e = tid; e < pn; e += nt) {
    const int u = (int)(e / n), rr = (int)(e % n);
    cplx acc[EV_CB];
#pragma unroll
    for (int q = 0; q < EV_CB; q++) acc[q] = mk(0.0, 0.0);
    for (int m = 0; m <= kmax; m++) {
      const T z = Zb[(size_t)u * nn + rr + (size_t)m * n];
#pragma unroll
      for (int q = 0; q < EV_CB; q++)
        if (s_col[q] >= 0) acc[q] = acc[q] + z * xcol(q, u)[m];
    }
#pragma unroll
    for (int q = 0; q < EV_CB; q++)
      if (s_col[q] >= 0) scol(q, u)[rr] = acc[q];  // s is no longer needed: it holds v
  }
  __syncthreads();
  cplx* Vb = P.V + (size_t)b * p * nn;
  for (int w = warp; w < EV_CB * p; w += nt >> 5) {
    const int q = w / p, u = w % p, c = s_col[q];
    if (c < 0) continue;
    const bool pair = s_top[q] > c;
    const cplx* v = scol(q, u);
    if (!ev_finish_column(n, lane, [&](int rr) { return v[rr]; }, Vb + (size_t)u * nn + (size_t)c * n,
                          pair ? Vb + (size_t)u * nn + (size_t)(c + 1) * n : nullptr, realT && !pair) &&
        lane == 0)
      P.info[b] = 2;
  }
}

// Global mode, after the host's GEMMs: Wre/Wim [2][p][m][n] hold Z_u X_u; one warp per (slot, u).
template <class T>
__global__ void __launch_bounds__(128) eigvecs_finish_kernel(EigvecParams P, const double* Wv) {
  const int n = P.n, p = P.p, lane = threadIdx.x & 31;
  const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (w >= P.m * p || P.info[0] == 1) return;
  const int slot = w / p, u = w % p;
  const int c = P.cols[slot];
  if (c < 0) return;
  const size_t nn = (size_t)n * n;
  const T* T0 = (const T*)P.T + (size_t)(P.left ? p - 1 : 0) * nn;
  const bool realT = sizeof(T) == sizeof(double);
  const bool pair = realT && c + 1 < n && !is_zero(T0[(c + 1) + (size_t)c * n]);
  const double* wr = Wv + ((size_t)u * P.m + slot) * n;
  const double* wi = wr + (size_t)p * P.m * n;
  if (!ev_finish_column(n, lane, [&](int rr) { return mk(wr[rr], wi[rr]); }, P.V + (size_t)u * nn + (size_t)c * n,
                        pair ? P.V + (size_t)u * nn + (size_t)(c + 1) * n : nullptr, realT && !pair) &&
      lane == 0)
    P.info[0] = 2;
}

}  // namespace psd
