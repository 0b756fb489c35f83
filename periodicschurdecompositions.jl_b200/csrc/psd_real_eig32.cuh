// Eigenvalue-only real periodic QR for small problems (n <= 32, p >= 3): ONE WARP PER PROBLEM.
//
// This is the B200 fast path of BASELINE config 2 (p=8, N=32, wantT=wantZ=false).  It
// implements the same iteration as periodic_qr_cta (PeriodicSchurDecompositions.jl:322-1096
// with wantT=false: updates restricted to the active window l..i, :675-678) but is organised
// around the hardware instead of around the reference's loop nest:
//
//  * lane L owns row L and column L of every factor; a 2- or 3-element reflector is applied
//    from the left by "column lanes" and from the right by "row lanes", so every update is
//    lane-local and no reduction is ever needed inside a sweep;
//  * a sweep is a flat sequence of chain links
//        H1(k) -> factor p -> factor p-1 -> ... -> factor 2 -> H1(k+1) -> ...
//    Each link's reflectors are computed redundantly by all lanes IN REGISTERS from the 3x3
//    diagonal block of its matrix (prefetched from shared memory one slot earlier) and the
//    previous link's reflectors, so the serial dependency chain contains no shuffle and no
//    shared-memory access; the 3-reflector of link t and the 2-reflector of link t-1 are
//    computed in the same slot (two independent dependency chains = ILP), and the row/column
//    updates of link t-1 ("bulk") are applied lane-parallel in that slot as well; with the
//    period fixed at compile time (p >= 4, the headline instantiation) the bulk runs two links
//    behind instead, so that it no longer waits for the 2-reflector of the same slot
//    (sweep_lag2);
//  * reflectors are kept un-normalised, H = I + g u u^T with g = -2/(u^T u): one rsqrt and
//    one reciprocal (MUFU seed + Newton steps) instead of dlarfg's sqrt + three divisions
//    (householder.jl:66-108); orthogonality of H depends only on g, not on the accuracy of
//    the norm; u^T u / 2 = |x|^2 + |x0| |x|, so the reciprocal's seed is taken from the rsqrt
//    SEED while the rsqrt is still being refined (refl_u);
//  * the factors live in shared memory in packed form (upper triangle + kl subdiagonals,
//    column c at offset c(c+1)/2 + kl*c): 36.4 KB per p=8,N=32 problem instead of 64 KB,
//    i.e. 6 resident problems per SM instead of 3, and both the column-lane and the row-lane
//    access patterns are bank-conflict free (triangular numbers mod 16 are a permutation);
//  * band quantities of the product (hdiag/hsub/hsup, :474-529) live in registers, one row
//    per lane, and the deflation scan (:531-585) is a single ballot.
//
// Indices in this file are 0-based.
#pragma once
#include <type_traits>

#include "psd_device.cuh"

namespace psd {

__host__ __device__ inline int pk_off(int kl, int c) { return c * (c + 1) / 2 + kl * c; }
__host__ __device__ inline int pk_size(int kl, int n) { return n * (n + 1) / 2 + kl * n; }
// doubles per packed problem: H1 with 3 subdiagonals (Hessenberg + bulge), others with 1
__host__ __device__ inline int pk_problem_size(int n, int p) {
  return pk_size(3, n) + (p - 1) * pk_size(1, n);
}

// Stride between packed problems: the factors plus one slot holding the power-of-two exponent E
// by which the product was scaled down (every factor is normalised to max |entry| in [0.5, 1) by
// an exact power of two before the iteration, because the un-normalised reflectors
// H = I + g u u^T square the entries; eigenvalues are multiplied by 2^E at the end).
// The slots behind the factors hold the state that travels between the occupancy phases of the
// iteration (see rpqr_eig32_kernel_t): [0] E, [1] current bottom index i (-1: finished or failed),
// [2] iterations left of the shared budget (:442-443), [3] iterations used so far.
constexpr int PK_STATE = 4;
__host__ __device__ inline int pk_problem_stride(int n, int p) { return pk_problem_size(n, p) + PK_STATE; }

struct EigParams {
  int n, p;
  long long batch;
  int maxitfac;
  const double* packed;  // [batch][pk_problem_stride(n, p)]
  double* packed_next;   // [batch][pk_problem_stride(stop, p)] or nullptr (last phase)
  int n_full;            // order of the original problems (row stride of eig)
  int stop;              // this phase works while the bottom index i >= stop
  int first_phase;       // state slots [1..3] are not set yet: start at i = n-1 with the full budget
  double* eig;           // [batch][n_full][2]
  int* info;
  int* iters;
  unsigned long long* counter;
  int force_safe;  // debug: skip the branch-free first attempt
};

PSD_DEV double shfl_d(double v, int src) { return __shfl_sync(0xffffffffu, v, src); }

// MUFU-seeded reciprocal square root / reciprocal with two Newton steps (~20-bit seeds).
PSD_DEV double fast_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double hx = 0.5 * x;
  double e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  return y;
}
PSD_DEV double fast_rcp(double x) {
  double y;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  double e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  e = fma(-x, y, 1.0);
  y = fma(y, e, y);
  return y;
}

// rare path of refl_u: zero tail (H = I, householder.jl:76-78) or out-of-range magnitudes,
// handled with an exact power-of-two prescale as dlarfg's sfmin loop does (:80-100).
struct ReflOut {
  double beta, u0, g;
};
template <int M>
__device__ __noinline__ ReflOut refl_u_slow(double x0, double x1, double x2) {
  ReflOut o;
  const double amax = fmax(fabs(x1), (M == 3) ? fabs(x2) : 0.0);
  if (amax == 0.0) {
    o.u0 = 0.0;
    o.g = 0.0;
    o.beta = x0;
    return o;
  }
  const double m = fmax(amax, fabs(x0));
  const double s = pow2_rescale(m);
  const double al = x0 * s, y1 = x1 * s, y2 = (M == 3) ? x2 * s : 0.0;
  const double nrm = sqrt(fma(al, al, fma(y1, y1, y2 * y2)));
  const double beta = -copysign(nrm, al);
  const double w0 = al - beta;
  o.u0 = w0 / s;
  o.g = (-2.0 * s) * (s / fma(w0, w0, fma(y1, y1, y2 * y2)));
  o.beta = beta / s;
  return o;
}

// Un-normalised reflector from (x0, x1[, x2]):  H = I + g u u^T, u = (x0 - beta, x1, x2),
// H x = beta e1.  Returns beta; g = 0 means H = I.
// SAFE = false: branch-free (so that the two reflector chains of a slot and the bulk updates
// can be interleaved by the instruction scheduler); magnitudes outside the range in which
// the squares are representable set `bad`, and the problem is then redone with SAFE = true,
// whose rare path rescales exactly like dlarfg (householder.jl:80-100).
template <int M, bool SAFE>
PSD_DEV double refl_u(double x0, double x1, double x2, double& u0, double& g, bool& bad) {
  const double ssq = (M == 3) ? fma(x1, x1, x2 * x2) : x1 * x1;
  const double nn = fma(x0, x0, ssq);
  const bool ok = (ssq > 1e-290 && nn < 1e290);
  if (SAFE) {
    if (!ok) {
      const ReflOut o = refl_u_slow<M>(x0, x1, x2);
      u0 = o.u0;
      g = o.g;
      return o.beta;
    }
  } else {
    bad = bad || (!ok && ssq != 0.0);
  }
#ifndef PSD_REFL_SERIAL
  // u'u / 2 = nn + |x0| nrm (with nrm^2 = nn), so g = -1 / (nn + |x0| nrm) needs no w0, and the
  // reciprocal seed can be taken from the 20-bit rsqrt seed while the rsqrt is still being
  // refined; its own Newton steps then use the exact denominator.  Shortens the dependent chain
  // of a reflector from ~175 to ~125 cycles.
  double r, y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(nn));
  const double ax = fabs(x0);
  {
    const double d0 = fma(nn * r, ax, nn);
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d0));
  }
  const double hx = 0.5 * nn;
  double e = fma(-hx * r, r, 0.5);
  r = fma(r, e, r);
  e = fma(-hx * r, r, 0.5);
  r = fma(r, e, r);
  const double nrm = nn * r;
  const double dd = fma(nrm, ax, nn);
  double f = fma(-dd, y, 1.0);
  y = fma(y, f, y);
  f = fma(-dd, y, 1.0);
  y = fma(y, f, y);
  const double gg = -y;
  const double beta = -copysign(nrm, x0);
  const double w0 = x0 - beta;
#else
  const double nrm = nn * fast_rsqrt(nn);
  const double beta = -copysign(nrm, x0);
  const double w0 = x0 - beta;
  const double gg = -2.0 * fast_rcp(fma(w0, w0, ssq));
#endif
  if (SAFE) {
    u0 = w0;
    g = gg;
    return beta;
  }
  // zero tail: H = I (householder.jl:76-78)
  u0 = ok ? w0 : 0.0;
  g = ok ? gg : 0.0;
  return ok ? beta : x0;
}

// State carried along the chain of links (all values identical in every lane).
struct ChainState {
  double u0, u1, u2, g, beta;           // 3-reflector of the previous link
  double c0, c1, h;                     // 2-reflector of the link before the previous one
  double n01, n02, n11, n12, n21, n22;  // columns 1,2 of N = X * P3 of the previous link
  double x00, x01, x02, x10, x11, x12, x22;  // diagonal block prefetched for the current link
};

// A part: N = X * (I + g u u^T); returns the first column (source of this link's 3-reflector)
// and stores columns 1,2 for the B part one slot later.
PSD_DEV void chain_A(const ChainState& c, double& s0, double& s1, double& s2, double& m01,
                     double& m02, double& m11, double& m12, double& m21, double& m22) {
  const double d0 = c.g * fma(c.x02, c.u2, fma(c.x01, c.u1, c.x00 * c.u0));
  const double d1 = c.g * fma(c.x12, c.u2, fma(c.x11, c.u1, c.x10 * c.u0));
  const double d2 = c.g * (c.x22 * c.u2);
  s0 = fma(d0, c.u0, c.x00);
  s1 = fma(d1, c.u0, c.x10);
  s2 = d2 * c.u0;
  m01 = fma(d0, c.u1, c.x01);
  m02 = fma(d0, c.u2, c.x02);
  m11 = fma(d1, c.u1, c.x11);
  m12 = fma(d1, c.u2, c.x12);
  m21 = d2 * c.u1;
  m22 = fma(d2, c.u2, c.x22);
}

// B part: 2-reflector of the previous (factor) link from its N, the 2-reflector before it
// and its own 3-reflector.
template <bool SAFE>
PSD_DEV double chain_B(const ChainState& c, double& b0, double& b1, double& bh, bool& bad) {
  const double e0 = c.h * fma(c.n02, c.c1, c.n01 * c.c0);
  const double e1 = c.h * fma(c.n12, c.c1, c.n11 * c.c0);
  const double e2 = c.h * fma(c.n22, c.c1, c.n21 * c.c0);
  const double m01 = fma(e0, c.c0, c.n01);
  const double m11 = fma(e1, c.c0, c.n11);
  const double m21 = fma(e2, c.c0, c.n21);
  const double f1 = c.g * fma(c.u2, m21, fma(c.u1, m11, c.u0 * m01));
  const double y0 = fma(f1, c.u1, m11);
  b1 = fma(f1, c.u2, m21);
  return refl_u<2, SAFE>(y0, b1, 0.0, b0, bh, bad);
}

// Row pass (right-multiplication by the previous link's reflectors) on a packed matrix at
// shared-memory index `base`: columns q..q+2 at packed offsets of0..of2, rows l..rmax,
// KL subdiagonals of storage.  FULLSTORE: store column q for every row (H1) instead of only
// above the diagonal (triangular factors, whose column q below the diagonal is the bulge that
// the next column pass overwrites with (beta, 0)).
template <int KL, bool HAS2>
PSD_DEV void row_pass(double* sm, int base, int of0, int of1, int of2, int q, int r, int l, int rmax,
                      bool c2, double u0, double u1, double u2, double g, double b0, double b1,
                      double bh) {
  // branch-free: lanes outside l..rmax compute on a clamped (valid) row and do not store
  const bool act = (r >= l && r <= rmax);
  const int rr = min(r, rmax);
  const bool e0x = (KL == 3) || (rr <= q + 1);
  const int o2 = c2 ? of2 : of1;
  double a0 = sm[base + of0 + (e0x ? rr : 0)];
  double a1 = sm[base + of1 + rr];
  double a2 = sm[base + o2 + rr];
  a0 = e0x ? a0 : 0.0;
  a2 = c2 ? a2 : 0.0;
  const double sa = g * fma(a2, u2, fma(a1, u1, a0 * u0));
  a0 = fma(sa, u0, a0);
  a1 = fma(sa, u1, a1);
  a2 = fma(sa, u2, a2);
  if (HAS2) {
    const double sb = bh * fma(a2, b1, a1 * b0);
    a1 = fma(sb, b0, a1);
    a2 = fma(sb, b1, a2);
  }
  if (act && ((KL == 3) || r < q)) sm[base + of0 + r] = a0;
  if (act) sm[base + of1 + r] = a1;
  if (act && c2) sm[base + of2 + r] = a2;
}

// Column pass (left-multiplication) on a triangular factor: column q <- (beta, 0), column
// q+1 <- (.., beta2, 0), columns > q+1 regular.
PSD_DEV void col_pass_tri(double* sm, int base, int ocj, int q, int r, int i, bool c2, double u0,
                          double u1, double u2, double g, double beta, double b0, double b1,
                          double bh, double beta2) {
  const bool act = (r >= q && r <= i);
  const int a = base + ocj + q;  // rows q.. of this lane's column (valid storage for r >= q)
  const int as = act ? a : base;  // inactive lanes read a harmless valid location
  double a0 = sm[as], a1 = sm[as + 1], a2 = sm[as + (c2 ? 2 : 1)];
  a2 = c2 ? a2 : 0.0;
  const double sa = g * fma(u2, a2, fma(u1, a1, u0 * a0));
  a0 = fma(sa, u0, a0);
  a1 = fma(sa, u1, a1);
  a2 = fma(sa, u2, a2);
  const double sb = bh * fma(b1, a2, b0 * a1);
  const bool d0 = (r == q), d1 = (r == q + 1);
  a0 = d0 ? beta : a0;
  a1 = d0 ? 0.0 : (d1 ? beta2 : fma(sb, b0, a1));
  a2 = d1 ? 0.0 : fma(sb, b1, a2);
  if (act) {
    sm[a] = a0;
    sm[a + 1] = a1;
  }
  if (act && c2 && !d0) sm[a + 2] = a2;
}

// Column pass on H1 with the H1-link's 3-reflector: columns q..i regular, column q-1 <-
// (beta, 0, 0) (the annihilated bulge), unless this is the first step of the sweep.
PSD_DEV void col_pass_h1(double* sm, int oc1, int q, int r, int i, int l, bool c2, double u0,
                         double u1, double u2, double g, double beta) {
  const bool reg = (r >= q && r <= i);
  const bool src = (r == q - 1 && q > l);
  const int a = oc1 + q;  // valid storage for r >= q-1 (3 subdiagonals)
  const int as = (reg || src) ? a : 0;
  double a0 = sm[as], a1 = sm[as + 1], a2 = sm[as + (c2 ? 2 : 1)];
  a2 = c2 ? a2 : 0.0;
  const double sa = g * fma(u2, a2, fma(u1, a1, u0 * a0));
  a0 = src ? beta : fma(sa, u0, a0);
  a1 = src ? 0.0 : fma(sa, u1, a1);
  a2 = src ? 0.0 : fma(sa, u2, a2);
  if (reg || src) {
    sm[a] = a0;
    sm[a + 1] = a1;
  }
  if ((reg || src) && c2) sm[a + 2] = a2;
}

// Both reflectors of one link, kept until its row/column passes ("bulk") run.  The H1 link has
// no 2-reflector; its bulk uses u, g and beta only.
struct LinkRefl {
  double u0, u1, u2, g, beta;
  double b0, b1, bh, beta2;
};

// 3x3 diagonal block of a link, prefetched one slot before its A part.
struct Blk {
  double x00, x01, x02, x10, x11, x12, x22;
};

// Block of triangular factor at `hb`, rows/columns k..k+2 (k..k+1 when C2 is false).
template <bool C2>
PSD_DEV Blk prefetch_tri(const double* sm, int hb, int t1a, int t1b, int t1c, int k) {
  Blk y;
  y.x00 = sm[hb + t1a + k];
  y.x01 = sm[hb + t1b + k];
  y.x10 = 0.0;
  y.x11 = sm[hb + t1b + k + 1];
  y.x02 = C2 ? sm[hb + t1c + k] : 0.0;
  y.x12 = C2 ? sm[hb + t1c + k + 1] : 0.0;
  y.x22 = C2 ? sm[hb + t1c + k + 2] : 0.0;
  return y;
}

// Block of the link H1(k+1): rows k+1..k+3, columns k..k+2 of H1 (only needed while k+2 <= i).
PSD_DEV Blk prefetch_h1(const double* sm, int t3a, int t3b, int t3c, int k, int i) {
  Blk y;
  const bool r3 = (k + 3 <= i);
  y.x00 = sm[t3a + k + 1];
  y.x01 = sm[t3b + k + 1];
  y.x02 = sm[t3c + k + 1];
  y.x10 = sm[t3a + k + 2];
  y.x11 = sm[t3b + k + 2];
  y.x12 = sm[t3c + k + 2];
  y.x22 = sm[t3c + (r3 ? k + 3 : k + 1)];
  y.x22 = r3 ? y.x22 : 0.0;
  return y;
}

PSD_DEV void set_block(ChainState& c, const Blk& y) {
  c.x00 = y.x00; c.x01 = y.x01; c.x02 = y.x02; c.x10 = y.x10; c.x11 = y.x11; c.x12 = y.x12;
  c.x22 = y.x22;
}

// Double-shift sweep over the window l..i with the bulk lagging TWO links behind the chain, for
// a period P >= 4 fixed at compile time.  The slot of link t (chain order H1(k), factor P, ...,
// factor 2, H1(k+1), ...) runs three independent streams:
//   * the A part and 3-reflector of link t (the loop-carried chain);
//   * the B part (2-reflector) of link t-1;
//   * the bulk of link t-2: column pass on its matrix M(t-2), row pass on M(t-1).
// The slot also prefetches the block of link t+1 from M(t+1) before its bulk.  Lag rule: compared
// with the one-link lag of the generic sweep, the only update that moves behind a prefetch is the
// bulk of link t-2 behind the prefetch of M(t+1) in slot t.  It writes M(t-2) and M(t-1), and links
// P apart share a matrix, so with P >= 4 it touches no prefetched entry:
//   * factor links: the block of factor j at step k still has pending only the row pass of link
//     t (folded by chain_A / chain_B, as before); the passes of step k-1 on factor j, the column
//     pass of factor j (k-1) (rows k-1..k+1) and the row pass of factor j+1 (k-1), or of H1(k-1)
//     for j = P (columns k-1..k+1), ran P-3 and P-2 slots before the prefetch;
//   * the H1 link: the block of H1(k+1) is read in the factor-2 slot of step k (slot P-1 of the
//     step), after the column pass of H1(k) (slot 2, needs P - 1 > 2) and the row pass of
//     factor 2 (k-1) (slot 1); the row pass of factor 2 (k) is folded by chain_A / chain_B.
// At P = 3 the column pass of M(t-2) = M(t+1) would hit rows k, k+1 of the prefetched block, so
// smaller periods keep the generic sweep.  Every stored element and every chain value therefore
// gets the same operations as in the generic sweep; only their order across slots differs.
// The factor loop is fully unrolled (prefetch sources and packed offsets are resolved per slot)
// and the last step of the sweep (k = i-1, the only one with k+2 > i) has its own instantiation.
template <bool SAFE, int P>
PSD_DEV void sweep_lag2(double* sm, const int szh1, const int sj, const int l, const int i,
                        const int r, const int ocj, const int oc1, const double v0, const double v1,
                        const double v2, bool& bad) {
  static_assert(P >= 4, "the two-link lag needs a period of at least 4");
  ChainState c;
  c.c0 = c.c1 = c.h = 0.0;
  LinkRefl d;  // reflectors of the link whose bulk is pending (link t-2 at the start of slot t)
  int t1a = pk_off(1, l), t1b = pk_off(1, l + 1), t1c = pk_off(1, l + 2);
  int t3a = pk_off(3, l), t3b = pk_off(3, l + 1), t3c = pk_off(3, l + 2);
  // previous step's offsets: the bulks of factors 3 and 2 run in the first two slots of a step
  int p1a = 0, p1b = 0, p1c = 0, p3a = 0, p3b = 0, p3c = 0;
  auto step = [&](const int k, auto c2tag) {
    constexpr bool C2 = decltype(c2tag)::value;  // k + 2 <= i
    const int rm2 = C2 ? k + 2 : k + 1;           // min(k + 2, i)
    double s0, s1, s2, m01, m02, m11, m12, m21, m22, nu0, ng, nbeta;
    Blk y;
    // =============== slot H1(k): bulk of factor 3 (k-1), B part of factor 2 (k-1) ===============
    __syncwarp();
    y = prefetch_tri<C2>(sm, szh1 + (P - 2) * sj, t1a, t1b, t1c, k);
    if (k > l) {
      double b0, b1, bh;
      const double beta2 = chain_B<SAFE>(c, b0, b1, bh, bad);
      row_pass<1, true>(sm, szh1, p1a, p1b, p1c, k - 1, r, l, k + 1, true, d.u0, d.u1, d.u2, d.g,
                        d.b0, d.b1, d.bh);
      col_pass_tri(sm, szh1 + sj, ocj, k - 1, r, i, true, d.u0, d.u1, d.u2, d.g, d.beta, d.b0, d.b1,
                   d.bh, d.beta2);
      chain_A(c, s0, s1, s2, m01, m02, m11, m12, m21, m22);
      d = LinkRefl{c.u0, c.u1, c.u2, c.g, c.beta, b0, b1, bh, beta2};
    } else {
      s0 = v0; s1 = v1; s2 = v2;
    }
    nbeta = refl_u<3, SAFE>(s0, s1, s2, nu0, ng, bad);
    set_block(c, y);
    c.u0 = nu0; c.u1 = s1; c.u2 = s2; c.g = ng; c.beta = nbeta;
    // =============== slot factor P: bulk of factor 2 (k-1) ===============
    __syncwarp();
    y = prefetch_tri<C2>(sm, szh1 + (P - 3) * sj, t1a, t1b, t1c, k);
    if (k > l) {
      row_pass<3, true>(sm, 0, p3a, p3b, p3c, k - 1, r, l, rm2, true, d.u0, d.u1, d.u2, d.g, d.b0,
                        d.b1, d.bh);
      col_pass_tri(sm, szh1, ocj, k - 1, r, i, true, d.u0, d.u1, d.u2, d.g, d.beta, d.b0, d.b1, d.bh,
                   d.beta2);
    }
    chain_A(c, s0, s1, s2, m01, m02, m11, m12, m21, m22);
    nbeta = refl_u<3, SAFE>(s0, s1, s2, nu0, ng, bad);
    d.u0 = c.u0; d.u1 = c.u1; d.u2 = c.u2; d.g = c.g; d.beta = c.beta;  // H1(k)
    set_block(c, y);
    c.c0 = 0.0; c.c1 = 0.0; c.h = 0.0;  // the H1 link has no 2-reflector
    c.u0 = nu0; c.u1 = s1; c.u2 = s2; c.g = ng; c.beta = nbeta;
    c.n01 = m01; c.n02 = m02; c.n11 = m11; c.n12 = m12; c.n21 = m21; c.n22 = m22;
    // ====== slots factor P-1 .. 2: B part of factor j+1, bulk of factor j+2 (H1(k) for j = P-1) ======
#pragma unroll
    for (int j = P - 1; j >= 2; j--) {
      __syncwarp();
      if (j > 2)
        y = prefetch_tri<C2>(sm, szh1 + (j - 3) * sj, t1a, t1b, t1c, k);
      else if (C2)
        y = prefetch_h1(sm, t3a, t3b, t3c, k, i);
      double b0, b1, bh;
      const double beta2 = chain_B<SAFE>(c, b0, b1, bh, bad);
      if (j == P - 1) {
        row_pass<1, false>(sm, szh1 + (P - 2) * sj, t1a, t1b, t1c, k, r, l, rm2, C2, d.u0, d.u1, d.u2,
                           d.g, 0.0, 0.0, 0.0);
        col_pass_h1(sm, oc1, k, r, i, l, C2, d.u0, d.u1, d.u2, d.g, d.beta);
      } else {
        row_pass<1, true>(sm, szh1 + (j - 1) * sj, t1a, t1b, t1c, k, r, l, rm2, C2, d.u0, d.u1, d.u2,
                          d.g, d.b0, d.b1, d.bh);
        col_pass_tri(sm, szh1 + j * sj, ocj, k, r, i, C2, d.u0, d.u1, d.u2, d.g, d.beta, d.b0, d.b1,
                     d.bh, d.beta2);
      }
      chain_A(c, s0, s1, s2, m01, m02, m11, m12, m21, m22);
      nbeta = refl_u<3, SAFE>(s0, s1, s2, nu0, ng, bad);
      d = LinkRefl{c.u0, c.u1, c.u2, c.g, c.beta, b0, b1, bh, beta2};  // factor j+1
      if (j > 2 || C2) set_block(c, y);
      c.c0 = b0; c.c1 = b1; c.h = bh;
      c.u0 = nu0; c.u1 = s1; c.u2 = s2; c.g = ng; c.beta = nbeta;
      c.n01 = m01; c.n02 = m02; c.n11 = m11; c.n12 = m12; c.n21 = m21; c.n22 = m22;
    }
    p1a = t1a; p1b = t1b; p1c = t1c;
    p3a = t3a; p3b = t3b; p3c = t3c;
    t1a = t1b; t1b = t1c; t1c += (k + 3) + 1;
    t3a = t3b; t3b = t3c; t3c += (k + 3) + 3;
  };
  for (int k = l; k < i - 1; k++) step(k, std::true_type{});
  step(i - 1, std::false_type{});
  // flush, two drained links: B part of factor 2 and bulk of factor 3 at k = i-1 ...
  {
    __syncwarp();
    double b0, b1, bh;
    const double beta2 = chain_B<SAFE>(c, b0, b1, bh, bad);
    row_pass<1, true>(sm, szh1, p1a, p1b, p1c, i - 1, r, l, i, false, d.u0, d.u1, d.u2, d.g, d.b0,
                      d.b1, d.bh);
    col_pass_tri(sm, szh1 + sj, ocj, i - 1, r, i, false, d.u0, d.u1, d.u2, d.g, d.beta, d.b0, d.b1,
                 d.bh, d.beta2);
    d = LinkRefl{c.u0, c.u1, c.u2, c.g, c.beta, b0, b1, bh, beta2};
  }
  // ... then the bulk of factor 2 at k = i-1
  {
    __syncwarp();
    row_pass<3, true>(sm, 0, p3a, p3b, p3c, i - 1, r, l, i, false, d.u0, d.u1, d.u2, d.g, d.b0, d.b1,
                      d.bh);
    col_pass_tri(sm, szh1, ocj, i - 1, r, i, false, d.u0, d.u1, d.u2, d.g, d.beta, d.b0, d.b1, d.bh,
                 d.beta2);
  }
}

// Result of one problem: info >= 0 as documented; kNeedSafe = magnitudes left the range the
// branch-free reflector handles, redo with SAFE = true.
constexpr int kNeedSafe = -12345;

// LAG2P > 0: the period is LAG2P (>= 4) and the sweep is sweep_lag2<SAFE, LAG2P>; 0: the generic
// sweep below, for any p >= 3 at run time.
template <bool SAFE, int LAG2P>
__device__ __forceinline__ int rpqr_problem(double* sm, const int n, const int p, const int i0,
                                            const int ml0, const int stop, const int lane,
                                            double& lre_out, double& lim_out, int& niter_out,
                                            int& i_end, int& ml_end) {
  const int szh1 = pk_size(3, n), sj = pk_size(1, n);
  const int r = lane;
  // this lane's column offsets in the two packed layouts, and those of columns r+1, r+2
  const int oc1 = pk_off(3, r), ocj = pk_off(1, r);
  const int ocj1 = pk_off(1, r + 1), ocj2 = pk_off(1, r + 2);
  const int oc1p = pk_off(3, r + 1), oc1m = (r > 0) ? pk_off(3, r - 1) : 0;
  const double dat1 = 0.75, dat2 = -0.4375;
  const double ulp = DBL_EPSILON;
  const double ulpx = ulp * sqrt(sqrt(ulp));
  const double smlnum = DBL_MIN * ((double)n / ulp);
  bool bad = false;
    double lre = 0.0, lim = 0.0;  // eigenvalue r lives in lane r
    int info = 0, niter = 0;

    i_end = -1;
    ml_end = 0;
    if (n == 1) {
      double q = sm[0];
      for (int j = 2; j <= p; j++) q *= sm[szh1 + (j - 2) * sj];
      lre = q;
    } else {
      int i = i0;
      int maxitleft = ml0;
      while (i >= stop) {
        int l = 0;
        int its = 1;
        bool splitting = false;
        double hdiag = 0.0, hsub = 0.0, hsup = 0.0;
        while (its < maxitleft) {
          // ---- band of the product, one row per lane (:474-529) ----
          const bool act = (r >= l && r <= i);
          const bool h1b = act && (r + 1 <= i), h2b = act && (r + 2 <= i);
          double q0 = 1.0, q1 = 0.0, q2 = 0.0;
          if (act) {
            int hb = szh1;
            for (int j = 2; j <= p; j++, hb += sj) {
              if (h2b)
                q2 = q0 * sm[hb + ocj2 + r] + q1 * sm[hb + ocj2 + r + 1] + q2 * sm[hb + ocj2 + r + 2];
              if (h1b) q1 = q0 * sm[hb + ocj1 + r] + q1 * sm[hb + ocj1 + r + 1];
              q0 *= sm[hb + ocj + r];
            }
          }
          const double t0m = __shfl_up_sync(0xffffffffu, q0, 1);
          const double t1m = __shfl_up_sync(0xffffffffu, q1, 1);
          const double t2m = __shfl_up_sync(0xffffffffu, q2, 1);
          const double t0p = __shfl_down_sync(0xffffffffu, q0, 1);
          if (act) {
            const double hd = sm[oc1 + r];
            const double hu = (r < i) ? sm[oc1p + r] : 0.0;
            if (r > l) {
              const double hs = sm[oc1m + r];
              hsub = hs * t0m;
              hdiag = hs * t1m + hd * q0;
              if (r < i) hsup = hs * t2m + hd * q1 + hu * t0p;
            } else {
              hsub = 0.0;
              hdiag = hd * q0;
              if (r < i) hsup = hd * q1 + hu * t0p;
            }
          }
          // ---- negligible-subdiagonal search (:497-585): lane k tests H[k,k-1] ----
          {
            const double hh11 = __shfl_up_sync(0xffffffffu, hdiag, 1);
            const double hh12 = __shfl_up_sync(0xffffffffu, hsup, 1);
            const bool tst = (r >= l + 1 && r <= i);
            bool found = false;
            double tst1 = fabs(hh11) + fabs(hdiag);
            const unsigned zmask = __ballot_sync(0xffffffffu, tst && tst1 == 0.0 && fabs(hsub) > smlnum);
            if (zmask) {
              // opnorm(H1[l:i,l:i], 1) fallback (:536-538): column sums, then warp max
              double cs = 0.0;
              if (act)
                for (int rr = l; rr <= min(r + 1, i); rr++) cs += fabs(sm[oc1 + rr]);
              cs = warp_max(cs);
              if (tst1 == 0.0) tst1 = cs;
            }
            if (tst) {
              const double a21 = fabs(hsub);
              if (a21 <= smlnum) {
                found = true;
              } else if (a21 <= ulp * tst1) {
                const double a12 = fabs(hh12);
                const double ab = fmax(a21, a12), ba = fmin(a21, a12);
                const double d12 = fabs(hh11 - hdiag);
                const double aa = fmax(fabs(hdiag), d12), bb = fmin(fabs(hdiag), d12);
                const double st = aa + ab;
                found = ba * (ab / st) <= fmax(smlnum, ulpx * (bb * (aa / st)));
              }
            }
            const unsigned fm = __ballot_sync(0xffffffffu, found);
            if (i > l) {
              if (fm) l = 31 - __clz(fm);
            } else {
              l = i;
            }
          }
          if (l >= i - 1) {
            splitting = true;
            break;
          }
          // ---- shifts (:679-764) and first column of the shift polynomial (:766-803) ----
          double v0, v1, v2;
          {
            const double h11 = shfl_d(hdiag, l), h12 = shfl_d(hsup, l);
            const double h21 = shfl_d(hsub, l + 1), h22 = shfl_d(hdiag, l + 1);
            const double hs3 = shfl_d(hsub, l + 2);
            const double hdi = shfl_d(hdiag, i), hdi1 = shfl_d(hdiag, i - 1);
            const double hsi = shfl_d(hsub, i), hsi1 = shfl_d(hsub, i - 1);
            const double hpi1 = shfl_d(hsup, i - 1);
            double s;
            if (its == 10 || its % 10 == 0) {
              if (its == 10)
                s = fabs(h21) + fabs(hs3);
              else
                s = fabs(hsi) + fabs(hsi1);
              const double h44 = dat1 * s + ((its == 10) ? h11 : hdi);
              const double h33 = h44;
              const double h43h34 = dat2 * s * s;
              const double h44s = h44 - h11, h33s = h33 - h11;
              v0 = (h33s * h44s - h43h34) / h21 + h12;
              v1 = h22 - h11 - h33s - h44s;
              v2 = hs3;
            } else {
              double h44 = hdi, h33 = hdi1, h43 = hsi, h34 = hpi1;
              double rt1r, rt2r, rt1i, rt2i;
              s = fabs(h33) + fabs(h34) + fabs(h43) + fabs(h44);
              if (s == 0.0) {
                rt1r = rt2r = rt1i = rt2i = 0.0;
              } else {
                h33 /= s; h44 /= s; h34 /= s; h43 /= s;
                const double trc = (h33 + h44) * 0.5;
                const double disc = (h33 - trc) * (h44 - trc) - h34 * h43;
                const double rtdisc = sqrt(fabs(disc));
                if (disc >= 0.0) {
                  rt1r = trc * s; rt2r = rt1r; rt1i = rtdisc * s; rt2i = -rt1i;
                } else {
                  rt1r = trc + rtdisc;
                  rt2r = trc - rtdisc;
                  rt1r = (fabs(rt1r - h44) <= fabs(rt2r - h44)) ? (rt1r * s) : (rt2r * s);
                  rt2r = rt1r;
                  rt1i = rt2i = 0.0;
                }
              }
              s = fabs(h11 - rt2r) + fabs(rt2i) + fabs(h21);
              const double h21s = h21 / s;
              v0 = h21s * h12 + (h11 - rt1r) * ((h11 - rt2r) / s) - rt1i * (rt2i / s);
              v1 = h21s * (h11 + h22 - rt1r - rt2r);
              v2 = h21s * hs3;
            }
            s = fabs(v0) + fabs(v1) + fabs(v2);
            v0 /= s; v1 /= s; v2 /= s;
          }

          // ---- double-shift sweep restricted to the window l..i (:806-886) ----
          if constexpr (LAG2P > 0) {
            sweep_lag2<SAFE, LAG2P>(sm, szh1, sj, l, i, r, ocj, oc1, v0, v1, v2, bad);
          } else {
            ChainState c;
            c.c0 = c.c1 = c.h = 0.0;
            // packed offsets of columns k, k+1, k+2 in both layouts, kept incrementally:
            // T(kl,c+1) = T(kl,c) + c + 1 + kl
            int t1a = pk_off(1, l), t1b = pk_off(1, l + 1), t1c = pk_off(1, l + 2);
            int t3a = pk_off(3, l), t3b = pk_off(3, l + 1), t3c = pk_off(3, l + 2);
            // previous step's kl=3 offsets (row pass on H1 runs one step late)
            int p3a = 0, p3b = 0, p3c = 0;
            for (int k = l; k < i; k++) {
              const bool c2 = (k + 2 <= i);
              const int rm2 = min(k + 2, i);
              double s0, s1, s2, m01, m02, m11, m12, m21, m22;
              double y00, y01, y02, y10, y11, y12, y22;  // block prefetched for the next link
              // Each slot is ONE scheduling region: sync; prefetch the next link's block; B part
              // of the previous link; bulk of the previous link; A part + 3-reflector of this
              // link.  (Requires p >= 3 so that the prefetched block is not touched by the
              // bulk of the same slot.)
              // =============== slot H1(k) ===============
              __syncwarp();
              {
                const int hb = szh1 + (p - 2) * sj;  // factor p at position k
                const int o2 = c2 ? t1c : t1b;
                y00 = sm[hb + t1a + k];
                y01 = sm[hb + t1b + k];
                y02 = sm[hb + o2 + k];
                y11 = sm[hb + t1b + k + 1];
                y12 = sm[hb + o2 + k + 1];
                y22 = sm[hb + o2 + (c2 ? k + 2 : k + 1)];
                y10 = 0.0;
                y02 = c2 ? y02 : 0.0; y12 = c2 ? y12 : 0.0; y22 = c2 ? y22 : 0.0;
              }
              if (k > l) {
                double b0, b1, bh;
                const double beta2 = chain_B<SAFE>(c, b0, b1, bh, bad);
                // bulk of factor 2 at step k-1: row pass on H1, column pass on H2
                row_pass<3, true>(sm, 0, p3a, p3b, p3c, k - 1, r, l, min(k + 2, i), true, c.u0, c.u1,
                                  c.u2, c.g, b0, b1, bh);
                col_pass_tri(sm, szh1, ocj, k - 1, r, i, true, c.u0, c.u1, c.u2, c.g, c.beta, b0, b1,
                             bh, beta2);
                chain_A(c, s0, s1, s2, m01, m02, m11, m12, m21, m22);
              } else {
                s0 = v0; s1 = v1; s2 = v2;
              }
              double nu0, ng;
              double nbeta = refl_u<3, SAFE>(s0, s1, s2, nu0, ng, bad);
              c.x00 = y00; c.x01 = y01; c.x02 = y02; c.x10 = y10; c.x11 = y11; c.x12 = y12; c.x22 = y22;
              c.u0 = nu0; c.u1 = s1; c.u2 = s2; c.g = ng; c.beta = nbeta;
              // =============== slot factor p: bulk of H1(k) ===============
              __syncwarp();
              {
                const int hb = szh1 + (p - 2) * sj;
                const int hn = hb - sj;  // factor p-1 at position k
                const int o2 = c2 ? t1c : t1b;
                y00 = sm[hn + t1a + k];
                y01 = sm[hn + t1b + k];
                y02 = sm[hn + o2 + k];
                y11 = sm[hn + t1b + k + 1];
                y12 = sm[hn + o2 + k + 1];
                y22 = sm[hn + o2 + (c2 ? k + 2 : k + 1)];
                y02 = c2 ? y02 : 0.0; y12 = c2 ? y12 : 0.0; y22 = c2 ? y22 : 0.0;
                row_pass<1, false>(sm, hb, t1a, t1b, t1c, k, r, l, rm2, c2, c.u0, c.u1, c.u2, c.g, 0.0,
                                   0.0, 0.0);
                col_pass_h1(sm, oc1, k, r, i, l, c2, c.u0, c.u1, c.u2, c.g, c.beta);
                chain_A(c, s0, s1, s2, m01, m02, m11, m12, m21, m22);
                nbeta = refl_u<3, SAFE>(s0, s1, s2, nu0, ng, bad);
                c.x00 = y00; c.x01 = y01; c.x02 = y02; c.x10 = 0.0; c.x11 = y11; c.x12 = y12; c.x22 = y22;
                c.c0 = 0.0; c.c1 = 0.0; c.h = 0.0;  // the H1 link has no 2-reflector
                c.u0 = nu0; c.u1 = s1; c.u2 = s2; c.g = ng; c.beta = nbeta;
                c.n01 = m01; c.n02 = m02; c.n11 = m11; c.n12 = m12; c.n21 = m21; c.n22 = m22;
              }
              // =============== slots factor p-1 .. 2 ===============
              for (int j = p - 1; j >= 2; j--) {
                const int hb = szh1 + (j - 2) * sj;  // this link's matrix; previous link's is hb + sj
                __syncwarp();
                if (j > 2) {
                  const int hn = hb - sj;
                  const int o2 = c2 ? t1c : t1b;
                  y00 = sm[hn + t1a + k];
                  y01 = sm[hn + t1b + k];
                  y02 = sm[hn + o2 + k];
                  y10 = 0.0;
                  y11 = sm[hn + t1b + k + 1];
                  y12 = sm[hn + o2 + k + 1];
                  y22 = sm[hn + o2 + (c2 ? k + 2 : k + 1)];
                  y02 = c2 ? y02 : 0.0; y12 = c2 ? y12 : 0.0; y22 = c2 ? y22 : 0.0;
                } else {
                  // next link is H1(k+1): rows k+1..k+3, columns k..k+2 of H1
                  const bool r3 = (k + 3 <= i);
                  const int o2 = c2 ? t3c : t3b;
                  const int r2i = c2 ? k + 2 : k + 1;
                  y00 = sm[t3a + k + 1];
                  y01 = sm[t3b + k + 1];
                  y02 = sm[o2 + k + 1];
                  y10 = sm[t3a + r2i];
                  y11 = sm[t3b + r2i];
                  y12 = sm[o2 + r2i];
                  y22 = sm[o2 + (r3 ? k + 3 : k + 1)];
                  y02 = c2 ? y02 : 0.0; y10 = c2 ? y10 : 0.0; y11 = c2 ? y11 : 0.0;
                  y12 = c2 ? y12 : 0.0; y22 = r3 ? y22 : 0.0;
                }
                double b0, b1, bh;
                const double beta2 = chain_B<SAFE>(c, b0, b1, bh, bad);
                row_pass<1, true>(sm, hb, t1a, t1b, t1c, k, r, l, rm2, c2, c.u0, c.u1, c.u2, c.g, b0, b1,
                                  bh);
                col_pass_tri(sm, hb + sj, ocj, k, r, i, c2, c.u0, c.u1, c.u2, c.g, c.beta, b0, b1, bh,
                             beta2);
                chain_A(c, s0, s1, s2, m01, m02, m11, m12, m21, m22);
                nbeta = refl_u<3, SAFE>(s0, s1, s2, nu0, ng, bad);
                c.x00 = y00; c.x01 = y01; c.x02 = y02; c.x10 = y10; c.x11 = y11; c.x12 = y12; c.x22 = y22;
                c.c0 = b0; c.c1 = b1; c.h = bh;
                c.u0 = nu0; c.u1 = s1; c.u2 = s2; c.g = ng; c.beta = nbeta;
                c.n01 = m01; c.n02 = m02; c.n11 = m11; c.n12 = m12; c.n21 = m21; c.n22 = m22;
              }
              // advance the packed offsets to step k+1
              p3a = t3a; p3b = t3b; p3c = t3c;
              t1a = t1b; t1b = t1c; t1c += (k + 3) + 1;
              t3a = t3b; t3b = t3c; t3c += (k + 3) + 3;
            }
            // flush: B part and bulk of factor 2 at the last step k = i-1
            {
              __syncwarp();
              double b0, b1, bh;
              const double beta2 = chain_B<SAFE>(c, b0, b1, bh, bad);
              row_pass<3, true>(sm, 0, p3a, p3b, p3c, i - 1, r, l, i, false, c.u0, c.u1, c.u2, c.g, b0,
                                b1, bh);
              col_pass_tri(sm, szh1, ocj, i - 1, r, i, false, c.u0, c.u1, c.u2, c.g, c.beta, b0, b1, bh,
                           beta2);
            }
          }
          __syncwarp();
          if (!SAFE && bad) return kNeedSafe;
          its++;
        }  // QR iterations

        if (!splitting) {
          info = i + 1;  // "convergence failed at level i" (:891-893), 1-based level
          niter += its;
          break;
        }
        // ---- deflation (:895-934, wantT = false) ----
        if (l == i) {
          if (r == i) {
            lre = hdiag;
            lim = 0.0;
          }
        } else {
          double a = shfl_d(hdiag, i - 1), bq = shfl_d(hsup, i - 1);
          double cq = shfl_d(hsub, i), d = shfl_d(hdiag, i);
          double cs, sn, l1r, l1i, l2r, l2i;
          gs2x2(a, bq, cq, d, cs, sn, l1r, l1i, l2r, l2i);
          if (r == i - 1) {
            lre = l1r;
            lim = l1i;
          } else if (r == i) {
            lre = l2r;
            lim = l2i;
          }
        }
        maxitleft -= its;
        niter += its;
        i = l - 1;
      }
      i_end = i;
      ml_end = maxitleft;
    }
    lre_out = lre;
    lim_out = lim;
    niter_out = niter;
    return info;
}

extern __shared__ __align__(16) double psd_smem_eig[];

// NN, PP > 0 fix the order and period at compile time (the headline shape N = 32, p = 8 gets its
// own instantiation: packed offsets and strides fold into constants); 0 = taken from the params.
// The iteration runs in up to three OCCUPANCY PHASES.  With wantT = false everything right of /
// below the current bottom index i is dead, so a problem whose bottom index has dropped below
// `stop` only needs the leading stop x stop part of every factor - which is a PREFIX of each
// packed array (column c always occupies c+1+kl slots).  A phase therefore works on problems of
// order n while i >= stop, writes the prefixes plus the loop state to the next phase's buffer,
// and the next launch treats them as problems of order `stop` with a smaller shared-memory
// footprint: more resident warps per SM where the latency-bound chain needs them
// (p = 8: order 32 -> 6 warps/SM, 24 -> 10; from there on the register file caps it).  Measured
// gain on the headline shape: 8-10 % (the iteration is only partly latency-bound).
// NN, PP > 0 fix the order and period at compile time (packed offsets and strides fold into
// constants); 0 = taken from the params.
template <int NN, int PP>
__device__ __forceinline__ void rpqr_eig32_body(const EigParams& P) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n = NN ? NN : P.n, p = PP ? PP : P.p;
  constexpr int kLag2P = (PP >= 4) ? PP : 0;  // compile-time period >= 4: sweep_lag2
  const int psize = pk_problem_size(n, p);
  const int stop = P.stop;
  double* sm = psd_smem_eig + (size_t)warp * psize;  // H1 at 0, factor j at szh1 + (j-2)*sj
  for (;;) {
    long long b = 0;
    if (lane == 0) b = (long long)atomicAdd(P.counter, 1ULL);
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= P.batch) break;
    const double* src = P.packed + (size_t)b * (psize + PK_STATE);
    const int escale = (int)src[psize];
    int i0, ml0, nit0;
    if (P.first_phase) {
      i0 = n - 1;
      ml0 = P.maxitfac * n;
      nit0 = 0;
    } else {
      i0 = (int)src[psize + 1];
      ml0 = (int)src[psize + 2];
      nit0 = (int)src[psize + 3];
    }
    double* nxt = P.packed_next ? P.packed_next + (size_t)b * pk_problem_stride(stop, p) : nullptr;
    if (i0 < 0) {  // finished or failed in an earlier phase
      if (nxt && lane == 0) nxt[pk_problem_size(stop, p) + 1] = -1.0;
      continue;
    }
    for (int e = lane; e < psize; e += 32) sm[e] = src[e];
    __syncwarp();
    double lre, lim;
    int niter, i_end, ml_end;
    int info = P.force_safe ? kNeedSafe
                            : rpqr_problem<false, kLag2P>(sm, n, p, i0, ml0, stop, lane, lre, lim, niter, i_end, ml_end);
    if (info == kNeedSafe) {
      // badly scaled problem: redo this phase with the exactly-rescaling reflector
      __syncwarp();
      for (int e = lane; e < psize; e += 32) sm[e] = src[e];
      __syncwarp();
      info = rpqr_problem<true, kLag2P>(sm, n, p, i0, ml0, stop, lane, lre, lim, niter, i_end, ml_end);
    }
    // eigenvalues found in this phase: indices i_end+1 .. i0 (all of 0..i0 after a failure, as the
    // single-phase kernel reports them)
    if (lane <= i0 && (lane > i_end || info != 0)) {
      double* eg = P.eig + ((size_t)b * P.n_full + lane) * 2;
      eg[0] = scalbn(lre, escale);
      eg[1] = scalbn(lim, escale);
    }
    const bool more = (info == 0 && i_end >= 0 && nxt != nullptr);
    if (lane == 0) {
      if (!more) {
        P.info[b] = info;
        if (P.iters) P.iters[b] = nit0 + niter;
      }
    }
    if (nxt) {
      __syncwarp();
      if (more) {
        // prefixes of the packed factors = the leading stop x stop problem
        const int s3 = pk_size(3, stop), s1 = pk_size(1, stop);
        const int szh1 = pk_size(3, n), sj = pk_size(1, n);
        for (int e = lane; e < s3; e += 32) nxt[e] = sm[e];
        for (int j = 2; j <= p; j++)
          for (int e = lane; e < s1; e += 32) nxt[s3 + (j - 2) * s1 + e] = sm[szh1 + (j - 2) * sj + e];
      }
      if (lane == 0) {
        double* stt = nxt + pk_problem_size(stop, p);
        stt[0] = (double)escale;
        stt[1] = more ? (double)i_end : -1.0;
        stt[2] = (double)ml_end;
        stt[3] = (double)(nit0 + niter);
      }
    }
    __syncwarp();
  }
}


// At most 256 threads per CTA leaves ptxas up to 255 registers.  The <32,8> instantiation uses
// 254 (no spills): its order-32 phase is held to 6 warps per SM by shared memory, and 6 warps
// of 256 registers fit the register file with room to spare.
template <int NN, int PP>
__global__ void __launch_bounds__(256) rpqr_eig32_kernel_t(EigParams P) {
  rpqr_eig32_body<NN, PP>(P);
}
// Register-capped instantiations for the later, small-footprint occupancy phases.  The register
// file is split over the four SM sub-partitions (16K registers each), so 172 registers per thread
// allow only 2 warps per sub-partition (8 per SM); <= 168 allow 3 (12 per SM), <= 128 allow 4.
__global__ void __launch_bounds__(96, 4) rpqr_eig32_kernel_r168(EigParams P) { rpqr_eig32_body<0, 0>(P); }
__global__ void __launch_bounds__(128, 4) rpqr_eig32_kernel_r128(EigParams P) { rpqr_eig32_body<0, 0>(P); }

}  // namespace psd
