// Building blocks of the GENERALIZED periodic Schur kernels (complex and real periodic QZ):
// scalar types, Givens generation, CTA-parallel rotation / reflector application, the
// "chase one rotation through every factor" primitive, and the generalized periodic
// Hessenberg-triangular reduction.
//
// Reference semantics restated here (file:line relative to the reference repository):
//   generalized.jl:988-1082   _phessenberg!(A, S)  Stage 1 (QR / RQ of factors p..2, applied to
//                             the neighbour factor and to Q[l]) and Stage 2 (Givens Hessenberg
//                             reduction of A_1, each rotation propagated through all factors)
//   generalized.jl:808-852    one step of the periodic QZ sweep (same propagation pattern)
//   generalized.jl:939-976    _safeprod
//   Julia stdlib givensAlgorithm / lmul!(Givens) / rmul!(., Givens') (LAPACK xLARTG semantics,
//   source not under the reference tree): [c s; -conj(s) c] [f; g] = [r; 0], c real.
//
// Execution model (same as psd_device.cuh): one CTA owns one periodic problem; scalar decisions
// are computed redundantly in registers by every thread from values read after a CTA barrier;
// row / column updates are dealt to the threads.
//
// The propagation primitive `chase_rotation` is organised around the hardware rather than the
// reference's loop nest: the rotation that enters factor l and the one that leaves it depend
// only on the 2x2 diagonal block of that factor, so the whole chain H_1 -> H_p -> ... -> H_2 ->
// H_1 is evaluated in registers (redundantly per thread), and every row/column update of every
// factor and of every Z_l touches memory that no other update of the same step reads.  A step
// therefore needs ONE CTA barrier instead of the 2p+1 of a literal transcription, and the
// loads of the next diagonal block overlap the updates of the current factor.
#pragma once
#include <cooperative_groups.h>

#include "psd_device.cuh"

namespace psd {

// ------------------------------------------------------------------------------------------
// complex128 (interleaved re, im: Julia ComplexF64 layout)
// ------------------------------------------------------------------------------------------
struct __align__(16) cplx {
  double x, y;
};
PSD_DEV cplx mk(double x, double y) {
  cplx r;
  r.x = x;
  r.y = y;
  return r;
}
PSD_DEV cplx operator+(cplx a, cplx b) { return mk(a.x + b.x, a.y + b.y); }
PSD_DEV cplx operator-(cplx a, cplx b) { return mk(a.x - b.x, a.y - b.y); }
PSD_DEV cplx operator-(cplx a) { return mk(-a.x, -a.y); }
PSD_DEV cplx operator*(cplx a, cplx b) {
  return mk(fma(a.x, b.x, -a.y * b.y), fma(a.x, b.y, a.y * b.x));
}
PSD_DEV cplx operator*(double a, cplx b) { return mk(a * b.x, a * b.y); }
PSD_DEV cplx operator*(cplx b, double a) { return mk(a * b.x, a * b.y); }
PSD_DEV cplx conj_(cplx a) { return mk(a.x, -a.y); }
PSD_DEV double conj_(double a) { return a; }
PSD_DEV double abs_(cplx a) { return hypot(a.x, a.y); }
PSD_DEV double abs_(double a) { return fabs(a); }
PSD_DEV double abs1_(cplx a) { return fabs(a.x) + fabs(a.y); }
PSD_DEV bool is_zero(cplx a) { return a.x == 0.0 && a.y == 0.0; }
PSD_DEV cplx scal2(cplx a, int k) { return mk(scalbn(a.x, k), scalbn(a.y, k)); }
PSD_DEV double scal2(double a, int k) { return scalbn(a, k); }
PSD_DEV bool is_zero(double a) { return a == 0.0; }
// Smith's complex division
PSD_DEV cplx operator/(cplx a, cplx b) {
  if (fabs(b.x) >= fabs(b.y)) {
    const double r = b.y / b.x, d = b.x + b.y * r;
    return mk((a.x + a.y * r) / d, (a.y - a.x * r) / d);
  }
  const double r = b.x / b.y, d = b.x * r + b.y;
  return mk((a.x * r + a.y) / d, (a.y * r - a.x) / d);
}
PSD_DEV cplx operator/(cplx a, double b) { return mk(a.x / b, a.y / b); }

template <class T>
struct Scalar;
template <>
struct Scalar<double> {
  static PSD_DEV double zero() { return 0.0; }
  static PSD_DEV double one() { return 1.0; }
  static PSD_DEV double from_real(double v) { return v; }
};
template <>
struct Scalar<cplx> {
  static PSD_DEV cplx zero() { return mk(0.0, 0.0); }
  static PSD_DEV cplx one() { return mk(1.0, 0.0); }
  static PSD_DEV cplx from_real(double v) { return mk(v, 0.0); }
};

// givensAlgorithm(f, g) -> (c, s, r), real: see givens_real in psd_device.cuh.
PSD_DEV void givens_t(double f, double g, double& c, double& s, double& r) {
  givens_real(f, g, c, s, r);
}
// complex (zlartg semantics): c = |f|/h, s = (f/|f|) conj(g)/h, r = (f/|f|) h, h = hypot(|f|,|g|)
PSD_DEV void givens_t(cplx f, cplx g, double& c, cplx& s, cplx& r) {
  if (is_zero(g)) {
    c = 1.0;
    s = mk(0.0, 0.0);
    r = f;
    return;
  }
  if (is_zero(f)) {
    const double ag = abs_(g);
    c = 0.0;
    s = conj_(g) / ag;
    r = mk(ag, 0.0);
    return;
  }
  double m = fmax(fmax(fabs(f.x), fabs(f.y)), fmax(fabs(g.x), fabs(g.y)));
  double sc = 1.0;
  if (m < 1e-140 || m > 1e140) sc = pow2_rescale(m);
  const cplx fs = sc * f, gs = sc * g;
  const double f2 = fma(fs.x, fs.x, fs.y * fs.y), g2 = fma(gs.x, gs.x, gs.y * gs.y);
  if (f2 == 0.0) {  // |f| negligible against |g| even after scaling
    const double ag = abs_(g);
    c = 0.0;
    s = conj_(g) / ag;
    r = mk(ag, 0.0);
    return;
  }
  const double h2 = f2 + g2;
  const double f1 = sqrt(f2), h = sqrt(h2);
  c = f1 / h;
  const double ifh = 1.0 / (f1 * h);
  s = (fs * conj_(gs)) * ifh;
  r = f * (h / f1);
}

// ------------------------------------------------------------------------------------------
// Problem context: factor l (1-based, INTERNAL rightwards order) at H + (l-1)*hs, leading
// dimension ldh; Z_l likewise.  S[l-1] is the internal signature (S[0] is always true).
// ------------------------------------------------------------------------------------------
template <class T>
struct GCtx {
  int n, p, tid, nt;
  T* H;
  long long hs;
  int ldh;
  T* Z;
  long long zs;
  int ldz;
  bool wantZ;
  bool zmap_left;
  const unsigned char* S;
  T* stage;     // 4 + 3(p-1) scalars of shared memory: diagonal blocks staged by chase_rotation
  T* stage_in;  // same size: the diagonal blocks of all factors, fetched with ONE parallel load
  long long* prof;  // phase time stamps (debug), or nullptr
  T* wvec;          // n scalars of shared memory: the reflector being applied (Stage 1)
  T* blk;           // blk_work_scalars(n) scalars of shared memory for the blocked Stage 1, or nullptr
  long long s2ws;   // offset (doubles) in dynamic shared memory of the s2_work_scalars(p) workspace of the
                    // windowed Stage 2, or -1
  long long qzws;   // same for the windowed double-shift sweep (qzw_work_doubles(p) doubles), or -1
  int deep_u;       // items in flight per thread in the deep variants (0: default)
  double* rots;     // 12(p+1) doubles of shared memory: rotation table of the deep (latency-hiding)
                    // chase variants, or nullptr to use the per-factor variants
  // Team mode (one large problem on the whole GPU, cooperative launch): every CTA runs the same
  // scalar control flow redundantly on values read from global memory after a grid barrier, the
  // row/column/Z updates are dealt to all threads of the grid (wtid of wnt), single-writer stores
  // are done by the leading CTA, and sync() is the grid barrier.  For a single CTA wtid = tid,
  // wnt = nt, lead = true and sync() is __syncthreads().
  int wtid, wnt;
  bool lead, team;
  PSD_DEV void sync() const {
    if (team)
      cooperative_groups::this_grid().sync();
    else
      __syncthreads();
  }
  PSD_DEV T* Hp(int l) const { return H + (long long)(l - 1) * hs; }
  PSD_DEV T* Zp(int l) const {
    int s = l;
    if (zmap_left && l > 1) s = p + 2 - l;  // Zr[l] = Z[p+2-l]  (generalized.jl:913-916)
    return Z + (long long)(s - 1) * zs;
  }
  PSD_DEV bool Sg(int l) const { return S[l - 1] != 0; }
};

#define PSD_GE(ptr, ld, r, c) (ptr)[((r)-1) + (size_t)((c)-1) * (ld)]

// rows (i1, i2) <- [c s; -conj(s) c] * rows, one column
template <class T>
PSD_DEV void rot_pair_rows(T* M, int ld, int i1, int i2, int col, double c, T s) {
  T* a = &PSD_GE(M, ld, i1, col);
  T* b = &PSD_GE(M, ld, i2, col);
  const T a1 = *a, a2 = *b;
  *a = c * a1 + s * a2;
  *b = c * a2 - conj_(s) * a1;
}
// columns (j1, j2) <- columns * Givens(j1,j2,c,s)', one row
template <class T>
PSD_DEV void rot_pair_cols(T* M, int ld, int j1, int j2, int row, double c, T s) {
  T* a = &PSD_GE(M, ld, row, j1);
  T* b = &PSD_GE(M, ld, row, j2);
  const T a1 = *a, a2 = *b;
  *a = c * a1 + conj_(s) * a2;
  *b = c * a2 - s * a1;
}

// Apply a list of independent 2-element rotations, dealt round-robin to the threads: item w is
// decoded by `item(w, a, b, c, s)` into two element pointers and the rotation
// (a, b) <- (c a + s b, c b - conj(s) a)   [rows: s; columns (right-multiplication by G'): conj(s)].
// All items touch disjoint memory, so BULK_U of them are loaded before any is stored: the loop is
// bound by memory latency (factors in L2 / HBM at the larger sizes), not by arithmetic.
constexpr int BULK_U = 4;
template <class T, class Item>
PSD_DEV void bulk_rot2(int tid, int nt, int total, Item&& item) {
  for (int w0 = tid; w0 < total; w0 += BULK_U * nt) {
    T* pa[BULK_U];
    T* pb[BULK_U];
    double cc[BULK_U];
    T ss[BULK_U], va[BULK_U], vb[BULK_U];
#pragma unroll
    for (int u = 0; u < BULK_U; u++) {
      const int w = w0 + u * nt;
      pa[u] = nullptr;
      if (w < total) item(w, pa[u], pb[u], cc[u], ss[u]);
    }
#pragma unroll
    for (int u = 0; u < BULK_U; u++)
      if (pa[u]) {
        va[u] = *pa[u];
        vb[u] = *pb[u];
      }
#pragma unroll
    for (int u = 0; u < BULK_U; u++)
      if (pa[u]) {
        *pa[u] = cc[u] * va[u] + ss[u] * vb[u];
        *pb[u] = cc[u] * vb[u] - conj_(ss[u]) * va[u];
      }
  }
}

// Deep variant for factors that live in L2 / HBM: the rotation of item w is looked up in a
// shared-memory table (rc[k], rs[k]) that covers ALL factors of one chase, so that a single pass
// with U independent items per thread in flight replaces p dependent passes (one memory round
// trip each).  item(w, a, off, k): element pair (a[0], a[off]), table entry k.
template <class T, int U, class Item>
PSD_DEV void bulk_rot2_tab(int tid, int nt, int total, const double* rc, const T* rs, Item&& item) {
  for (int w0 = tid; w0 < total; w0 += U * nt) {
    T* pa[U];
    int off[U], kk[U];
    T va[U], vb[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int w = w0 + u * nt;
      pa[u] = nullptr;
      if (w < total) item(w, pa[u], off[u], kk[u]);
    }
#pragma unroll
    for (int u = 0; u < U; u++)
      if (pa[u]) {
        va[u] = pa[u][0];
        vb[u] = pa[u][off[u]];
      }
#pragma unroll
    for (int u = 0; u < U; u++)
      if (pa[u]) {
        const double c = rc[kk[u]];
        const T s = rs[kk[u]];
        pa[u][0] = c * va[u] + s * vb[u];
        pa[u][off[u]] = c * vb[u] - conj_(s) * va[u];
      }
  }
}
// w -> (w / per, w % per) with a float reciprocal and a fix-up (w < 2^24)
PSD_DEV void split_index(int w, int per, float rper, int& q, int& r) {
  if (w >= (1 << 24)) {  // beyond the exact range of the float estimate
    q = w / per;
    r = w - q * per;
    return;
  }
  q = (int)((float)w * rper);
  r = w - q * per;
  if (r < 0) {
    q--;
    r += per;
  } else if (r >= per) {
    q++;
    r -= per;
  }
}

// ---- simple CTA-synchronous helpers (used on the rarely taken branches) -------------------
// lmul!(Givens(i1,i2,c,s), view(M, :, c0:c1)); barrier at the end
template <class T>
PSD_DEV void g_lmul(const GCtx<T>& cx, T* M, int ld, int i1, int i2, double c, T s, int c0, int c1) {
  for (int col = c0 + cx.wtid; col <= c1; col += cx.wnt) rot_pair_rows(M, ld, i1, i2, col, c, s);
  cx.sync();
}
// rmul!(view(M, r0:r1, :), Givens(j1,j2,c,s)'); barrier at the end
template <class T>
PSD_DEV void g_rmul(const GCtx<T>& cx, T* M, int ld, int j1, int j2, double c, T s, int r0, int r1) {
  for (int row = r0 + cx.wtid; row <= r1; row += cx.wnt) rot_pair_cols(M, ld, j1, j2, row, c, s);
  cx.sync();
}
// c, s, r = givensAlgorithm(M[fa], M[ga]); M[fa] = r; M[ga] = 0   (barrier-safe)
template <class T>
PSD_DEV void g_gen(const GCtx<T>& cx, T* M, int ld, int fr, int fc, int gr, int gc, double& c, T& s) {
  const T f = PSD_GE(M, ld, fr, fc), g = PSD_GE(M, ld, gr, gc);
  T r;
  givens_t(f, g, c, s, r);
  cx.sync();
  if (cx.lead && cx.tid == 0) {
    PSD_GE(M, ld, fr, fc) = r;
    PSD_GE(M, ld, gr, gc) = Scalar<T>::zero();
  }
  cx.sync();
}

// opnorm(view(M, r0:r1, c0:c1), 1), optionally of the upper triangle of the view (rare
// fallback of the deflation tolerances; serial, executed by every calling thread).
template <class T>
PSD_DEV double g_opnorm1(const T* M, int ld, int r0, int r1, int c0, int c1, bool upper) {
  double m = 0.0;
  for (int c = c0; c <= c1; c++) {
    double s = 0.0;
    const int rl = upper ? min(r1, r0 + (c - c0)) : r1;
    for (int r = r0; r <= rl; r++) s += abs_(PSD_GE(M, ld, r, c));
    m = fmax(m, s);
  }
  return m;
}

// One link of the rotation chain: the incoming rotation (ci, si) meets the 2x2 diagonal block
// [c00 c01; 0 c11] of a triangular factor (S = true: from the right, S = false: from the left);
// co, so is the rotation that restores the triangle and travels on, (cR, sR) the one acting on
// the block's column pair above it, (cL, sL) the one acting on its row pair to the right, m the
// updated block.
template <class T>
struct RotChain {
  double co, cR, cL;
  T so, sR, sL, m00, m01, m11;
};
// Rotation generation inside the chains.  Real: one reciprocal square root (MUFU seed + two Newton
// steps, full double precision) instead of a square root and three divisions; same sign convention
// as givens_real.  Complex: givens_t.
PSD_DEV double chain_rsqrt(double x) {
  double y;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
  const double hx = 0.5 * x;
  double e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  e = fma(-hx * y, y, 0.5);
  y = fma(y, e, y);
  return y;
}
PSD_DEV void givens_chain(double f, double g, double& c, double& s, double& r) {
  const double m = fmax(fabs(f), fabs(g));
  if (g == 0.0 || f == 0.0 || !(m > 1e-140 && m < 1e140)) {
    givens_real(f, g, c, s, r);
    return;
  }
  const double t = fma(f, f, g * g);
  const double y = chain_rsqrt(t);
  c = f * y;
  s = g * y;
  r = t * y;
  if (fabs(f) > fabs(g) && c < 0.0) {
    c = -c; s = -s; r = -r;
  }
}
PSD_DEV void givens_chain(cplx f, cplx g, double& c, cplx& s, cplx& r) { givens_t(f, g, c, s, r); }

template <class T>
PSD_DEV void rot_chain_step(bool sl, double ci, T si, T c00, T c01, T c11, RotChain<T>& o) {
  if (sl) {
    // block * G_in'  then  G_out * block
    const T n00 = ci * c00 + conj_(si) * c01;
    const T n01 = ci * c01 - si * c00;
    const T n10 = conj_(si) * c11;
    const T n11 = ci * c11;
    T r;
    givens_chain(n00, n10, o.co, o.so, r);
    o.m00 = r;
    o.m01 = o.co * n01 + o.so * n11;
    o.m11 = o.co * n11 - conj_(o.so) * n01;
    o.cR = ci; o.sR = si;
    o.cL = o.co; o.sL = o.so;
  } else {
    // G_in * block  then  block * Givens(j+1, j, co, conj(so))'  (rows rfirst..j only)
    const T n00 = ci * c00;
    const T n01 = ci * c01 + si * c11;
    const T n10 = -(conj_(si) * c00);
    const T n11 = ci * c11 - conj_(si) * c01;
    T r;
    givens_chain(n11, n10, o.co, o.so, r);
    o.m01 = o.co * n01 + o.so * n00;
    o.m00 = o.co * n00 - conj_(o.so) * n01;
    o.m11 = r;
    o.cL = ci; o.sL = si;
    o.so = -o.so;  // equivalent Givens(j, j+1, co, -so)  (generalized.jl:839-840)
    o.cR = o.co; o.sR = o.so;
  }
}

// ------------------------------------------------------------------------------------------
// chase_rotation: apply G1 = Givens(j, j+1, c1, s1) to H_1 from the left (columns h1c0..clast),
// propagate it through factors p..2 (generalized.jl:823-845 / :1045-1075), apply the rotation
// that comes out to H_1 from the right (rows rfirst..h1r1) and accumulate every rotation into
// the Z_l.  If zcol > 0 the generating pair of H_1 is overwritten: H_1[j,zcol] = r1,
// H_1[j+1,zcol] = 0.  For a factor with S = true the incoming rotation acts on its columns
// (rows rfirst..j+1) and the outgoing one on its rows (columns j+1..clast); with S = false the
// incoming one acts on rows (columns j..clast) and the outgoing one on columns (rows rfirst..j).
// Two barriers: one after the bulk updates (every thread has then consumed the diagonal blocks
// it read), one after the 2x2 diagonal blocks, staged in shared memory meanwhile, have been
// written back.  All threads of the CTA must call with identical arguments.
// ------------------------------------------------------------------------------------------
template <class T>
__device__ __noinline__ void chase_rotation(const GCtx<T>& cx, int j, double c1, T s1, int zcol, T r1, int h1c0,
                            int clast, int rfirst, int h1r1) {
  const int n = cx.n, p = cx.p, tid = cx.tid, nt = cx.nt;
  T* H1 = cx.Hp(1);
  const int ld = cx.ldh;
  // All 2x2 diagonal blocks (H_1: 4 entries at [0..3], factor l: 3 entries at 4+3(l-2)) are
  // fetched by one parallel load into shared memory: the chain below then costs one memory
  // latency per step instead of one per factor.
  {
    T* in = cx.stage_in;
    for (int e = tid; e < 4 + 3 * (p - 1); e += nt) {
      if (e < 4) {
        in[e] = PSD_GE(H1, ld, j + (e >> 1), j + (e & 1));
      } else {
        const int l = 2 + (e - 4) / 3, w = (e - 4) % 3;
        in[e] = PSD_GE(cx.Hp(l), ld, j + (w == 2 ? 1 : 0), j + (w == 0 ? 0 : 1));
      }
    }
    __syncthreads();
  }
  const T* bin = cx.stage_in;
  const T ha = bin[0], hb = bin[1], hc = bin[2], hd = bin[3];
  if (cx.rots) {
    // Deep variant: one thread walks the chain and publishes every rotation, then ONE bulk pass
    // covers the rows / columns / Z columns of all factors.
    T* rs = reinterpret_cast<T*>(cx.rots);
    double* rc = reinterpret_cast<double*>(rs + 3 * p);
    if (tid == 0) {
      double ci = c1;
      T si = s1;
      for (int l = p; l >= 2; l--) {
        RotChain<T> o;
        rot_chain_step<T>(cx.Sg(l), ci, si, bin[4 + 3 * (l - 2)], bin[5 + 3 * (l - 2)], bin[6 + 3 * (l - 2)], o);
        const int k = 3 * (l - 2);
        rc[k] = o.cR; rs[k] = conj_(o.sR);
        rc[k + 1] = o.cL; rs[k + 1] = o.sL;
        rc[k + 2] = o.co; rs[k + 2] = conj_(o.so);
        T* st = cx.stage + 4 + 3 * (l - 2);
        st[0] = o.m00; st[1] = o.m01; st[2] = o.m11;
        ci = o.co;
        si = o.so;
      }
      const int k = 3 * (p - 1);
      rc[k] = c1; rs[k] = s1;                // rows (j, j+1) of H_1
      rc[k + 1] = c1; rs[k + 1] = conj_(s1);  // columns (j, j+1) of Z_1
      rc[k + 2] = ci; rs[k + 2] = conj_(si);  // columns (j, j+1) of H_1
      const T a1 = c1 * ha + s1 * hc, b1 = c1 * hb + s1 * hd;
      const T a2 = c1 * hc - conj_(s1) * ha, b2 = c1 * hd - conj_(s1) * hb;
      cx.stage[0] = ci * a1 + conj_(si) * b1;
      cx.stage[1] = ci * b1 - si * a1;
      cx.stage[2] = ci * a2 + conj_(si) * b2;
      cx.stage[3] = ci * b2 - si * a2;
    }
    __syncthreads();
    const int nR = j - rfirst, nL = clast - (j + 1), nZ = cx.wantZ ? n : 0;
    const int per = nR + nL + nZ, nf = (p - 1) * per;
    const int nL1 = (clast - h1c0 + 1) - 2, nR1 = (h1r1 - rfirst + 1) - 2;
    const int total = nf + nL1 + nZ + nR1;
    const float rper = per > 0 ? 1.0f / (float)per : 0.0f;
    const int ldz = cx.ldz, k1 = 3 * (p - 1);
    auto deep_item = [&](int w, T*& a, int& off, int& k) {
      if (w < nf) {
        int f, r;
        split_index(w, per, rper, f, r);
        const int l = 2 + f;
        k = 3 * f;
        if (r < nR) {
          a = &PSD_GE(cx.Hp(l), ld, rfirst + r, j);
          off = ld;
        } else if (r < nR + nL) {
          a = &PSD_GE(cx.Hp(l), ld, j, j + 2 + (r - nR));
          off = 1;
          k += 1;
        } else {
          a = &PSD_GE(cx.Zp(l), ldz, 1 + (r - nR - nL), j);
          off = ldz;
          k += 2;
        }
      } else {
        int r = w - nf;
        if (r < nL1) {
          int col = h1c0 + r;
          if (col >= j) col += 2;
          a = &PSD_GE(H1, ld, j, col);
          off = 1;
          k = k1;
        } else if (r < nL1 + nZ) {
          a = &PSD_GE(cx.Zp(1), ldz, 1 + (r - nL1), j);
          off = ldz;
          k = k1 + 1;
        } else {
          int row = rfirst + (r - nL1 - nZ);
          if (row >= j) row += 2;
          a = &PSD_GE(H1, ld, row, j);
          off = ld;
          k = k1 + 2;
        }
      }
    };
    if (cx.deep_u == 8)
      bulk_rot2_tab<T, 8>(cx.wtid, cx.wnt, total, rc, rs, deep_item);
    else if (cx.deep_u == 2)
      bulk_rot2_tab<T, 2>(cx.wtid, cx.wnt, total, rc, rs, deep_item);
    else
      bulk_rot2_tab<T, 4>(cx.wtid, cx.wnt, total, rc, rs, deep_item);
    cx.sync();
    for (int l = 1 + tid; cx.lead && l <= p; l += nt) {
      if (l == 1) {
        PSD_GE(H1, ld, j, j) = cx.stage[0];
        PSD_GE(H1, ld, j, j + 1) = cx.stage[1];
        PSD_GE(H1, ld, j + 1, j) = cx.stage[2];
        PSD_GE(H1, ld, j + 1, j + 1) = cx.stage[3];
        if (zcol > 0) {
          PSD_GE(H1, ld, j, zcol) = r1;
          PSD_GE(H1, ld, j + 1, zcol) = Scalar<T>::zero();
        }
      } else {
        T* Hl = cx.Hp(l);
        const T* st = cx.stage + 4 + 3 * (l - 2);
        PSD_GE(Hl, ld, j, j) = st[0];
        PSD_GE(Hl, ld, j, j + 1) = st[1];
        PSD_GE(Hl, ld, j + 1, j) = Scalar<T>::zero();
        PSD_GE(Hl, ld, j + 1, j + 1) = st[2];
      }
    }
    cx.sync();
    return;
  }
  double ci = c1;
  T si = s1;
  T b00 = Scalar<T>::zero(), b01 = b00, b11 = b00;
  // Z_1 and the left-only part of H_1 (rotation G1); the overlap block is finished at the end
  {
    const int nL = (clast - h1c0 + 1) - 2;  // columns h1c0..clast without j, j+1
    const int nZ = cx.wantZ ? n : 0;
    T* Z1 = cx.wantZ ? cx.Zp(1) : nullptr;
    const int ldz = cx.ldz;
    bulk_rot2<T>(cx.wtid, cx.wnt, nL + nZ, [&](int w, T*& a, T*& b, double& c, T& s) {
      c = c1;
      if (w < nL) {
        int col = h1c0 + w;
        if (col >= j) col += 2;
        a = &PSD_GE(H1, ld, j, col);
        b = a + 1;
        s = s1;
      } else {
        a = &PSD_GE(Z1, ldz, 1 + (w - nL), j);
        b = a + ldz;
        s = conj_(s1);
      }
    });
  }
  for (int l = p; l >= 2; l--) {
    T* Hl = cx.Hp(l);
    b00 = bin[4 + 3 * (l - 2)];
    b01 = bin[5 + 3 * (l - 2)];
    b11 = bin[6 + 3 * (l - 2)];
    RotChain<T> rc_;
    rot_chain_step<T>(cx.Sg(l), ci, si, b00, b01, b11, rc_);
    const double co = rc_.co, cR = rc_.cR, cL = rc_.cL;
    const T so = rc_.so, sR = rc_.sR, sL = rc_.sL, m00 = rc_.m00, m01 = rc_.m01, m11 = rc_.m11;
    {
      const int nR = j - rfirst;  // rows rfirst..j-1
      const int nL = clast - (j + 1);  // columns j+2..clast
      const int nZ = cx.wantZ ? n : 0;
      T* Zl = cx.wantZ ? cx.Zp(l) : nullptr;
      const int ldz = cx.ldz;
      bulk_rot2<T>(cx.wtid, cx.wnt, nR + nL + nZ, [&](int w, T*& a, T*& b, double& c, T& s) {
        if (w < nR) {
          a = &PSD_GE(Hl, ld, rfirst + w, j);
          b = a + ld;
          c = cR;
          s = conj_(sR);
        } else if (w < nR + nL) {
          a = &PSD_GE(Hl, ld, j, j + 2 + (w - nR));
          b = a + 1;
          c = cL;
          s = sL;
        } else {
          a = &PSD_GE(Zl, ldz, 1 + (w - nR - nL), j);
          b = a + ldz;
          c = co;
          s = conj_(so);
        }
      });
      if (tid == 0) {
        T* st = cx.stage + 4 + 3 * (l - 2);
        st[0] = m00;
        st[1] = m01;
        st[2] = m11;
      }
    }
    ci = co;
    si = so;
  }
  // right-only rows of H_1 (rotation that came out of factor 2) and the overlap block
  {
    const int nR = (h1r1 - rfirst + 1) - 2;  // rows rfirst..h1r1 without j, j+1
    bulk_rot2<T>(cx.wtid, cx.wnt, nR, [&](int w, T*& a, T*& b, double& c, T& s) {
      int row = rfirst + w;
      if (row >= j) row += 2;
      a = &PSD_GE(H1, ld, row, j);
      b = a + ld;
      c = ci;
      s = conj_(si);
    });
    if (tid == 0) {
      // left with G1, then right with (ci, si)
      const T a1 = c1 * ha + s1 * hc, b1 = c1 * hb + s1 * hd;
      const T a2 = c1 * hc - conj_(s1) * ha, b2 = c1 * hd - conj_(s1) * hb;
      cx.stage[0] = ci * a1 + conj_(si) * b1;
      cx.stage[1] = ci * b1 - si * a1;
      cx.stage[2] = ci * a2 + conj_(si) * b2;
      cx.stage[3] = ci * b2 - si * a2;
    }
  }
  cx.sync();
  for (int l = 1 + tid; cx.lead && l <= p; l += nt) {
    if (l == 1) {
      PSD_GE(H1, ld, j, j) = cx.stage[0];
      PSD_GE(H1, ld, j, j + 1) = cx.stage[1];
      PSD_GE(H1, ld, j + 1, j) = cx.stage[2];
      PSD_GE(H1, ld, j + 1, j + 1) = cx.stage[3];
      if (zcol > 0) {
        PSD_GE(H1, ld, j, zcol) = r1;
        PSD_GE(H1, ld, j + 1, zcol) = Scalar<T>::zero();
      }
    } else {
      T* Hl = cx.Hp(l);
      const T* st = cx.stage + 4 + 3 * (l - 2);
      PSD_GE(Hl, ld, j, j) = st[0];
      PSD_GE(Hl, ld, j, j + 1) = st[1];
      PSD_GE(Hl, ld, j + 1, j) = Scalar<T>::zero();
      PSD_GE(Hl, ld, j + 1, j + 1) = st[2];
    }
  }
  cx.sync();
}

// ------------------------------------------------------------------------------------------
// Householder reflectors for Stage 1 (generalized.jl:1009-1028; geqrf!/gerqf! + ormqr!/ormrq!).
// H = I - tau w w^H.  Each warp recomputes the norm redundantly (no broadcast step).
// ------------------------------------------------------------------------------------------
PSD_DEV double sq_(double a) { return a * a; }
PSD_DEV double sq_(cplx a) { return fma(a.x, a.x, a.y * a.y); }
PSD_DEV double re_(double a) { return a; }
PSD_DEV double re_(cplx a) { return a.x; }
PSD_DEV double im_(double) { return 0.0; }
PSD_DEV double im_(cplx a) { return a.y; }
PSD_DEV double amax_(double a) { return fabs(a); }
PSD_DEV double amax_(cplx a) { return fmax(fabs(a.x), fabs(a.y)); }
PSD_DEV double rdiv_one(double d) { return 1.0 / d; }
PSD_DEV cplx rdiv_one(cplx d) { return Scalar<cplx>::one() / d; }

// Reflector from the m-vector x[k*inc], k = 0..m-1 (pivot first).  Returns false when H = I.
// On return: beta (new pivot value, real), tau, and tv such that w = (1, tv * x[1:]).
// For complex data with CONJ the reflector is built for conj(x) (row reflectors).
template <class T, bool CONJ>
PSD_DEV bool refl_vec(const T* x, long long inc, int m, int lane, double& beta, T& tau, T& tv) {
  double amax = 0.0;
  for (int k = 1 + lane; k < m; k += 32) amax = fmax(amax, amax_(x[k * inc]));
  amax = warp_max(amax);
  T alpha = x[0];
  if (CONJ) alpha = conj_(alpha);
  if (amax == 0.0 && im_(alpha) == 0.0) return false;
  const double mm = fmax(amax, amax_(alpha));
  double s = 1.0;
  if (mm < 1e-140 || mm > 1e140) s = pow2_rescale(mm);
  double ssq = 0.0;
  for (int k = 1 + lane; k < m; k += 32) ssq += sq_(s * x[k * inc]);
  ssq = warp_sum(ssq);
  const T al = s * alpha;
  const double b = -copysign(sqrt(sq_(al) + ssq), re_(al));
  // tau = (beta - alpha)/beta (complex: ((beta-ar)/beta, -ai/beta)); v = x[1:] / (alpha - beta)
  tau = (Scalar<T>::from_real(b) - al) * (1.0 / b);
  tv = s * rdiv_one(al - Scalar<T>::from_real(b));
  beta = b / s;
  return true;
}

// ---- reflector application with memory-level parallelism ------------------------------------
// The reflector w (w_0 = 1) is placed in shared memory once; every loop below then loads HH_U
// matrix entries before using any of them.  (A literal "d += a[r] * w[r]" loop that reads w from
// the matrix it updates is fully latency-exposed: the compiler must assume the stores alias it.)
constexpr int HH_U = 8;

// a[0], a[st], ..., a[(m-1) st]  <-  (I - coef w w^H)-type update of one row/column vector:
//   d = sum_r f(w_r) a_r;  a_r -= (coef d) g(w_r)
// RIGHT = true:  d = sum a_r w_r,        a_r -= (tau d) conj(w_r)     (A H,   one thread per row)
template <class T>
PSD_DEV void hh_right_one(T* a, long long st, int m, const T* w, T tau) {
  T d = Scalar<T>::zero();
  int r = 0;
  for (; r + HH_U <= m; r += HH_U) {
    T v[HH_U];
#pragma unroll
    for (int u = 0; u < HH_U; u++) v[u] = a[(long long)(r + u) * st];
#pragma unroll
    for (int u = 0; u < HH_U; u++) d = d + v[u] * w[r + u];
  }
  for (; r < m; r++) d = d + a[(long long)r * st] * w[r];
  d = tau * d;
  r = 0;
  for (; r + HH_U <= m; r += HH_U) {
    T v[HH_U];
#pragma unroll
    for (int u = 0; u < HH_U; u++) v[u] = a[(long long)(r + u) * st];
#pragma unroll
    for (int u = 0; u < HH_U; u++) a[(long long)(r + u) * st] = v[u] - d * conj_(w[r + u]);
  }
  for (; r < m; r++) a[(long long)r * st] = a[(long long)r * st] - d * conj_(w[r]);
}

// H' A on one column handled by a warp: a_r at a[r*st], r < m; d = conj(tau) sum conj(w_r) a_r;
// a_r -= d w_r.  Lanes stride over r; up to 4 strided chunks are loaded at once.
template <class T>
PSD_DEV void hh_left_warp(T* a, long long st, int m, const T* w, T tau, int lane) {
  T d = Scalar<T>::zero();
  for (int r = lane; r < m; r += 128) {
    T v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) v[u] = (r + 32 * u < m) ? a[(long long)(r + 32 * u) * st] : Scalar<T>::zero();
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (r + 32 * u < m) d = d + conj_(w[r + 32 * u]) * v[u];
  }
  if constexpr (sizeof(T) == sizeof(double)) {
    d = warp_sum(d);
  } else {
    d.x = warp_sum(d.x);
    d.y = warp_sum(d.y);
  }
  d = conj_(tau) * d;
  for (int r = lane; r < m; r += 128) {
    T v[4];
#pragma unroll
    for (int u = 0; u < 4; u++) v[u] = (r + 32 * u < m) ? a[(long long)(r + 32 * u) * st] : Scalar<T>::zero();
#pragma unroll
    for (int u = 0; u < 4; u++)
      if (r + 32 * u < m) a[(long long)(r + 32 * u) * st] = v[u] - d * w[r + 32 * u];
  }
}

// QR-type step on column k of Al (S[l] = true): annihilate Al[k+1:n, k]; apply H' to the
// remaining columns of Al, H to the neighbour factor (from the right if S[l-1], H' from the
// left otherwise) and to Q_l from the right.
template <class T>
PSD_DEV void stage1_qr_step(const GCtx<T>& cx, T* Al, T* Am, bool sm1, T* Ql, int k) {
  const int n = cx.n, ld = cx.ldh, tid = cx.tid, nt = cx.nt;
  const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int m = n - k + 1;
  T* xg = &PSD_GE(Al, ld, k, k);
  double beta;
  T tau, tv;
  if (!refl_vec<T, false>(xg, 1, m, lane, beta, tau, tv)) return;  // uniform over the CTA
  T* w = cx.wvec;  // w_0 = 1, w_r = tv x_r  (rows k..n)
  for (int r = tid; r < m; r += nt) w[r] = (r == 0) ? Scalar<T>::one() : tv * xg[r];
  __syncthreads();
  // (a) left on Al columns k+1..n and, when !S[l-1], on all columns of Am: one warp per column
  const int ncolA = n - k, ncolM = sm1 ? 0 : n;
  for (int c = warp; c < ncolA + ncolM; c += nw) {
    T* a = (c < ncolA) ? &PSD_GE(Al, ld, k, k + 1 + c) : &PSD_GE(Am, ld, k, 1 + (c - ncolA));
    hh_left_warp<T>(a, 1, m, w, tau, lane);
  }
  // (b) right on Am rows (if S[l-1]) and Q_l rows: one thread per row
  const int nM = sm1 ? n : 0, nQ = cx.wantZ ? n : 0;
  for (int c = tid; c < nM + nQ; c += nt) {
    if (c < nM)
      hh_right_one<T>(&PSD_GE(Am, ld, 1 + c, k), ld, m, w, tau);
    else
      hh_right_one<T>(&PSD_GE(Ql, cx.ldz, 1 + (c - nM), k), cx.ldz, m, w, tau);
  }
  __syncthreads();
  for (int r = tid; r < m; r += nt)
    PSD_GE(Al, ld, k + r, k) = (r == 0) ? Scalar<T>::from_real(beta) : Scalar<T>::zero();
  __syncthreads();
}

// RQ-type step on row k of Al (S[l] = false): annihilate Al[k, 1:k-1] with a reflector G acting
// on columns 1..k (pivot = column k); Al <- Al G (rows 1..k-1), neighbour factor Am <- Am G
// (if S[l-1]) or G' Am (otherwise), Q_l <- Q_l G.
template <class T>
PSD_DEV void stage1_rq_step(const GCtx<T>& cx, T* Al, T* Am, bool sm1, T* Ql, int k) {
  const int n = cx.n, ld = cx.ldh, tid = cx.tid, nt = cx.nt;
  const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int m = k;
  // vector conj(Al[k, k]), conj(Al[k, k-1]), ..., conj(Al[k, 1]): pivot first, stride -ld
  T* xg = &PSD_GE(Al, ld, k, k);
  const long long inc = -(long long)ld;
  double beta;
  T tau, tv;
  if (!refl_vec<T, true>(xg, inc, m, lane, beta, tau, tv)) return;
  T* w = cx.wvec;  // w_0 = 1 (column k), w_r = tv conj(x_r) (column k-r)
  for (int r = tid; r < m; r += nt) w[r] = (r == 0) ? Scalar<T>::one() : tv * conj_(xg[r * inc]);
  __syncthreads();
  // (a) right on rows: Al rows 1..k-1, Am rows 1..n (if S[l-1]), Q_l rows 1..n
  const int nA = k - 1, nM = sm1 ? n : 0, nQ = cx.wantZ ? n : 0;
  for (int c = tid; c < nA + nM + nQ; c += nt) {
    if (c < nA)
      hh_right_one<T>(&PSD_GE(Al, ld, 1 + c, k), -(long long)ld, m, w, tau);
    else if (c < nA + nM)
      hh_right_one<T>(&PSD_GE(Am, ld, 1 + (c - nA), k), -(long long)ld, m, w, tau);
    else
      hh_right_one<T>(&PSD_GE(Ql, cx.ldz, 1 + (c - nA - nM), k), -(long long)cx.ldz, m, w, tau);
  }
  // (b) left G' on all columns of Am rows 1..k (if !S[l-1]): one warp per column
  if (!sm1)
    for (int c = warp; c < n; c += nw) hh_left_warp<T>(&PSD_GE(Am, ld, k, 1 + c), -1, m, w, tau, lane);
  __syncthreads();
  for (int r = tid; r < m; r += nt)
    PSD_GE(Al, ld, k, k - r) = (r == 0) ? Scalar<T>::from_real(beta) : Scalar<T>::zero();
  __syncthreads();
}

// ------------------------------------------------------------------------------------------
// Blocked Stage 1 (compact WY), used when the factors live in global memory.
//
// The unblocked steps above make two passes over every matrix per reflector; at N = 256..512 with
// all SMs busy that traffic dominates the whole decomposition (profiles/r1_c5_ncu_full_raw.csv).
// Here S1_NB reflectors are generated on a panel held in shared memory, their compact-WY form
// I - V T V^H (dlarft, forward columnwise) is built, and the three big matrices are updated with
// two passes per PANEL: S1_NB fused multiply-adds per element loaded.
//
// The RQ-type factors (S[l] = false) reuse the QR code through the view
//     B(r, c) = conj(A(n-1-c, n-1-r)):   A = R Q   <=>   B = Qb Rb,   Q = J Qb^H J
// (J = reversal), so  A_{l-1} Q^H = (A_{l-1} J) Qb J  and  Q A_{l-1} = J Qb^H (J A_{l-1})  are the
// same right / left block applications on index-reversed views.
// ------------------------------------------------------------------------------------------
constexpr int S1_NB = 16;

template <class T>
struct BlkView {
  T* p;              // element (0, 0)
  long long rs, cs;  // element (r, c) at p[r*rs + c*cs]
  bool cj;           // stored value is the conjugate of the view's value
};
template <class T>
PSD_DEV T bv_get(const BlkView<T>& v, int r, int c) {
  const T x = v.p[r * v.rs + c * v.cs];
  return v.cj ? conj_(x) : x;
}
template <class T>
PSD_DEV void bv_set(const BlkView<T>& v, int r, int c, T x) {
  v.p[r * v.rs + c * v.cs] = v.cj ? conj_(x) : x;
}
template <class T>
PSD_DEV T wsum_t(T d) {
  if constexpr (sizeof(T) == sizeof(double)) {
    return warp_sum(d);
  } else {
    d.x = warp_sum(d.x);
    d.y = warp_sum(d.y);
    return d;
  }
}

// shared-memory workspace of the blocked Stage 1: Vs[kb][m] (column q of V at Vs + q*m), Ts, Gs
template <class T>
struct BlkWork {
  T* Vs;
  T* Ts;  // [S1_NB][S1_NB], T(t,q) at Ts[t + q*S1_NB]
  T* Gs;  // Gram matrix V^H V, same layout
  T* taus;
};
__host__ __device__ inline long long blk_work_scalars(int n) { return (long long)n * S1_NB + 2 * S1_NB * S1_NB + S1_NB; }

// QR of the panel B[c0:n, c0:c0+kb] (view), reflectors left in W.Vs as an explicit unit lower
// trapezoid (m x kb), T in W.Ts; the panel of B is overwritten with R (exact zeros below).
template <class T>
PSD_DEV void blk_panel_qr(const GCtx<T>& cx, const BlkView<T>& B, int c0, int kb, const BlkWork<T>& W) {
  const int n = cx.n, tid = cx.tid, nt = cx.nt;
  const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int m = n - c0;
  T* Ps = W.Vs;
  for (int e = tid; e < m * kb; e += nt) Ps[e] = bv_get(B, c0 + e % m, c0 + e / m);
  __syncthreads();
  for (int q = 0; q < kb; q++) {
    const int len = m - q;
    T* x = Ps + (size_t)q * m + q;
    double beta;
    T tau, tv;
    const bool nontrivial = refl_vec<T, false>(x, 1, len, lane, beta, tau, tv);
    if (nontrivial) {
      T* w = cx.wvec;
      for (int r = tid; r < len; r += nt) w[r] = (r == 0) ? Scalar<T>::one() : tv * x[r];
      __syncthreads();
      for (int c = q + 1 + warp; c < kb; c += nw) hh_left_warp<T>(Ps + (size_t)c * m + q, 1, len, w, tau, lane);
      for (int r = tid; r < len; r += nt) x[r] = (r == 0) ? Scalar<T>::from_real(beta) : w[r];
      if (tid == 0) W.taus[q] = tau;
    } else if (tid == 0) {
      W.taus[q] = Scalar<T>::zero();
    }
    __syncthreads();
  }
  // R back to the view, then the explicit V (unit diagonal, zeros above)
  for (int e = tid; e < m * kb; e += nt) {
    const int r = e % m, q = e / m;
    bv_set(B, c0 + r, c0 + q, (r <= q) ? Ps[e] : Scalar<T>::zero());
  }
  __syncthreads();
  for (int e = tid; e < kb * kb; e += nt) {
    const int r = e % kb, q = e / kb;
    if (r <= q) Ps[(size_t)q * m + r] = (r == q) ? Scalar<T>::one() : Scalar<T>::zero();
  }
  __syncthreads();
  // Gram matrix G(t, q) = V_t^H V_q, t < q (one warp per pair), then T column by column
  for (int pr = warp; pr < kb * kb; pr += nw) {
    const int t = pr % kb, q = pr / kb;
    if (t >= q) continue;
    T d = Scalar<T>::zero();
    for (int r = q + lane; r < m; r += 32) d = d + conj_(Ps[(size_t)t * m + r]) * Ps[(size_t)q * m + r];
    d = wsum_t(d);
    if (lane == 0) W.Gs[t + q * S1_NB] = d;
  }
  __syncthreads();
  for (int q = 0; q < kb; q++) {
    if (tid < q) {
      T acc = Scalar<T>::zero();
      for (int sidx = tid; sidx < q; sidx++) acc = acc + W.Ts[tid + sidx * S1_NB] * W.Gs[sidx + q * S1_NB];
      W.Ts[tid + q * S1_NB] = -(W.taus[q] * acc);
    } else if (tid == q) {
      W.Ts[q + q * S1_NB] = W.taus[q];
    }
    __syncthreads();
  }
}

// M <- M (I - V T V^H), M(row, c) at M[row*rs + c*cs], c = 0..m-1; one thread per row.
// CJ: use conj(V), conj(T) (the operand is stored conjugated).
template <class T, bool CJ>
PSD_DEV void blk_apply_right(const GCtx<T>& cx, T* M, long long rs, long long cs, int nrows, int m, int kb,
                             const BlkWork<T>& W) {
  const T* Vs = W.Vs;
  for (int row = cx.tid; row < nrows; row += cx.nt) {
    T* a = M + row * rs;
    T acc[S1_NB];
#pragma unroll
    for (int q = 0; q < S1_NB; q++) acc[q] = Scalar<T>::zero();
    for (int c = 0; c < m; c += 4) {
      T v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) v[u] = (c + u < m) ? a[(c + u) * cs] : Scalar<T>::zero();
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (c + u < m) {
#pragma unroll
          for (int q = 0; q < S1_NB; q++)
            if (q < kb) {
              const T vv = Vs[(size_t)q * m + c + u];
              acc[q] = acc[q] + v[u] * (CJ ? conj_(vv) : vv);
            }
        }
    }
    T w2[S1_NB];
#pragma unroll
    for (int q = 0; q < S1_NB; q++) {
      T z = Scalar<T>::zero();
#pragma unroll
      for (int t = 0; t < S1_NB; t++)
        if (t <= q && q < kb) {
          const T tt = W.Ts[t + q * S1_NB];
          z = z + acc[t] * (CJ ? conj_(tt) : tt);
        }
      w2[q] = z;
    }
    for (int c = 0; c < m; c += 4) {
      T v[4];
#pragma unroll
      for (int u = 0; u < 4; u++) v[u] = (c + u < m) ? a[(c + u) * cs] : Scalar<T>::zero();
#pragma unroll
      for (int u = 0; u < 4; u++)
        if (c + u < m) {
          T z = v[u];
#pragma unroll
          for (int q = 0; q < S1_NB; q++)
            if (q < kb) {
              const T vv = Vs[(size_t)q * m + c + u];
              z = z - w2[q] * (CJ ? vv : conj_(vv));
            }
          a[(c + u) * cs] = z;
        }
    }
  }
}

// M <- (I - V T^H V^H) M, M(r, col) at M[r*rs + col*cs], r = 0..m-1; one warp per column.
template <class T, bool CJ>
PSD_DEV void blk_apply_left(const GCtx<T>& cx, T* M, long long rs, long long cs, int ncols, int m, int kb,
                            const BlkWork<T>& W) {
  const int lane = cx.tid & 31, warp = cx.tid >> 5, nw = cx.nt >> 5;
  const T* Vs = W.Vs;
  for (int col = warp; col < ncols; col += nw) {
    T* a = M + col * cs;
    T acc[S1_NB];
#pragma unroll
    for (int q = 0; q < S1_NB; q++) acc[q] = Scalar<T>::zero();
    for (int r = lane; r < m; r += 64) {
      const T v0 = a[r * rs];
      const bool h1 = r + 32 < m;
      const T v1 = h1 ? a[(r + 32) * rs] : Scalar<T>::zero();
#pragma unroll
      for (int q = 0; q < S1_NB; q++)
        if (q < kb) {
          const T x0 = Vs[(size_t)q * m + r];
          acc[q] = acc[q] + (CJ ? x0 : conj_(x0)) * v0;
          if (h1) {
            const T x1 = Vs[(size_t)q * m + r + 32];
            acc[q] = acc[q] + (CJ ? x1 : conj_(x1)) * v1;
          }
        }
    }
#pragma unroll
    for (int q = 0; q < S1_NB; q++)
      if (q < kb) acc[q] = wsum_t(acc[q]);
    T w2[S1_NB];
#pragma unroll
    for (int q = 0; q < S1_NB; q++) {
      T z = Scalar<T>::zero();
#pragma unroll
      for (int t = 0; t < S1_NB; t++)
        if (t <= q && q < kb) {  // (T^H acc)_q = sum_{t <= q} conj(T(t, q)) acc_t
          const T tt = W.Ts[t + q * S1_NB];
          z = z + (CJ ? tt : conj_(tt)) * acc[t];
        }
      w2[q] = z;
    }
    for (int r = lane; r < m; r += 64) {
      const bool h1 = r + 32 < m;
      T v0 = a[r * rs];
      T v1 = h1 ? a[(r + 32) * rs] : Scalar<T>::zero();
#pragma unroll
      for (int q = 0; q < S1_NB; q++)
        if (q < kb) {
          const T x0 = Vs[(size_t)q * m + r];
          v0 = v0 - (CJ ? conj_(x0) : x0) * w2[q];
          if (h1) {
            const T x1 = Vs[(size_t)q * m + r + 32];
            v1 = v1 - (CJ ? conj_(x1) : x1) * w2[q];
          }
        }
      a[r * rs] = v0;
      if (h1) a[(r + 32) * rs] = v1;
    }
  }
}

// Stage 1 for factor l with the blocked scheme (matrices in global memory, leading dimension ld).
template <class T>
PSD_DEV void stage1_blocked(const GCtx<T>& cx, int l, const BlkWork<T>& W) {
  const int n = cx.n, ld = cx.ldh, ldz = cx.ldz;
  T* Al = cx.Hp(l);
  T* Am = cx.Hp(l - 1);
  T* Ql = cx.wantZ ? cx.Zp(l) : nullptr;
  const bool sl = cx.Sg(l), sm1 = cx.Sg(l - 1);
  BlkView<T> B;
  if (sl) {
    B.p = Al; B.rs = 1; B.cs = ld; B.cj = false;
  } else {
    B.p = Al + (n - 1) + (size_t)(n - 1) * ld; B.rs = -(long long)ld; B.cs = -1; B.cj = true;
  }
  for (int c0 = 0; c0 < n - 1; c0 += S1_NB) {
    const int kb = min(S1_NB, n - 1 - c0), m = n - c0, c1 = c0 + kb;
    blk_panel_qr(cx, B, c0, kb, W);
    // trailing columns of the factor itself: B[c0:, c1:] <- Qb^H B[c0:, c1:]
    if (n - c1 > 0) {
      T* M = B.p + c0 * B.rs + c1 * B.cs;
      if (B.cj)
        blk_apply_left<T, true>(cx, M, B.rs, B.cs, n - c1, m, kb, W);
      else
        blk_apply_left<T, false>(cx, M, B.rs, B.cs, n - c1, m, kb, W);
    }
    if (sl) {
      // A_{l-1} <- A_{l-1} Qb  or  Qb^H A_{l-1};   Q_l <- Q_l Qb
      if (sm1)
        blk_apply_right<T, false>(cx, Am + (size_t)c0 * ld, 1, ld, n, m, kb, W);
      else
        blk_apply_left<T, false>(cx, Am + c0, 1, ld, n, m, kb, W);
      if (Ql) blk_apply_right<T, false>(cx, Ql + (size_t)c0 * ldz, 1, ldz, n, m, kb, W);
    } else {
      // Q^H = J Qb J:  A_{l-1} <- (A_{l-1} J) Qb J  or  J Qb^H (J A_{l-1});   Q_l <- (Q_l J) Qb J
      if (sm1)
        blk_apply_right<T, false>(cx, Am + (size_t)(n - 1 - c0) * ld, 1, -(long long)ld, n, m, kb, W);
      else
        blk_apply_left<T, false>(cx, Am + (n - 1 - c0), -1, ld, n, m, kb, W);
      if (Ql) blk_apply_right<T, false>(cx, Ql + (size_t)(n - 1 - c0) * ldz, 1, -(long long)ldz, n, m, kb, W);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// Windowed Stage 2 (factors in global memory).
//
// The rotations that zero column jc of H_1 act on the adjacent row pairs (i-1, i), i = n ... jc+2.
// They are processed S2_K at a time.  Inside one batch everything the rotation chains depend on
// lives in the (kb+1) x (kb+1) diagonal windows of the triangular factors and in column jc of
// H_1, so one warp walks the kb chains on copies of those windows in shared memory and records
// every rotation in a table.  Left and right multiplications commute, so outside the windows a
// factor only sees a SEQUENCE of column rotations (rows above the window), a sequence of row
// rotations (columns right of the window), and Z_l a sequence of column rotations: each thread
// loads the kb+1 adjacent entries of one row / column, applies the whole sequence in registers
// and stores them back.  Compared with one pass per rotation this halves the traffic, makes the
// row updates contiguous (kb+1 entries of a column instead of one pair) and needs four barriers
// per batch instead of three per rotation.  H_1 gets all left rotations first, then all right ones.
// ------------------------------------------------------------------------------------------
constexpr int S2_K = 16, S2_W = S2_K + 1;
__host__ __device__ inline long long s2_work_scalars(int p) {
  return (long long)(p - 1) * S2_W * S2_W + S2_W + 2LL * S2_K * (3 * (p - 1) + 3) + 8;
}

// Explicit global-memory accesses (the factor pointers travel through GCtx as generic pointers).
PSD_DEV double ldg_(const double* p) {
  double v;
  asm volatile("ld.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
PSD_DEV cplx ldg_(const cplx* p) {
  cplx v;
  asm volatile("ld.global.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
  return v;
}
PSD_DEV void stg_(double* p, double v) { asm volatile("st.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }
PSD_DEV void stg_(cplx* p, cplx v) {
  asm volatile("st.global.v2.f64 [%0], {%1, %2};" ::"l"(p), "d"(v.x), "d"(v.y) : "memory");
}

// x[q] <-> ptr[(q - (S2_W - W)) * stride], q = S2_W - W .. S2_W - 1 (W = kb + 1); rotation t acts
// on the pair (x[S2_W-1-t], x[S2_W-t]) as (a, b) <- (c a + s b, c b - conj(s) a); its entry is at
// index (t-1)*E of the shared-memory tables rc / rs.  FULL: kb == S2_K, straight-line code.
template <class T, bool FULL>
PSD_DEV void s2_apply_seq(T* ptr, long long stride, int kb, const double* rc, const T* rs, int E) {
  const int sh = FULL ? 0 : S2_W - (kb + 1);
  T x[S2_W];
  if (FULL) {
    double c[S2_K];
    T sv[S2_K];
#pragma unroll
    for (int q = 0; q < S2_W; q++) x[q] = ldg_(ptr + (long long)q * stride);
#pragma unroll
    for (int t = 0; t < S2_K; t++) {
      c[t] = rc[t * E];
      sv[t] = rs[t * E];
    }
#pragma unroll
    for (int t = 1; t <= S2_K; t++) {
      const T a = x[S2_W - 1 - t], b = x[S2_W - t];
      x[S2_W - 1 - t] = c[t - 1] * a + sv[t - 1] * b;
      x[S2_W - t] = c[t - 1] * b - conj_(sv[t - 1]) * a;
    }
#pragma unroll
    for (int q = 0; q < S2_W; q++) stg_(ptr + (long long)q * stride, x[q]);
    return;
  }
#pragma unroll
  for (int q = 0; q < S2_W; q++)
    if (q >= sh) x[q] = ldg_(ptr + (long long)(q - sh) * stride);
#pragma unroll
  for (int t = 1; t <= S2_K; t++)
    if (t <= kb) {
      const double c = rc[(t - 1) * E];
      const T sv = rs[(t - 1) * E];
      const T a = x[S2_W - 1 - t], b = x[S2_W - t];
      x[S2_W - 1 - t] = c * a + sv * b;
      x[S2_W - t] = c * b - conj_(sv) * a;
    }
#pragma unroll
  for (int q = 0; q < S2_W; q++)
    if (q >= sh) stg_(ptr + (long long)(q - sh) * stride, x[q]);
}

extern __shared__ __align__(16) double psd_smem_cq[];

// ws_off: offset (in doubles) of the workspace inside the kernel's dynamic shared memory; taking
// the address from the array itself keeps the accesses in the shared state space (LDS / STS).
template <class T>
PSD_DEV void stage2_windowed(const GCtx<T>& cx, long long ws_off) {
  const int n = cx.n, p = cx.p, tid = cx.tid, nt = cx.nt, ld = cx.ldh, ldz = cx.ldz;
  const int lane = tid & 31, warp = tid >> 5;
  const int E = 3 * (p - 1) + 3;  // table entries per rotation: (R, L, Z) per factor 2..p, then H1 left, Z1, H1 right
  T* Dw = reinterpret_cast<T*>(psd_smem_cq + ws_off);  // [(p-1)][S2_W][S2_W], column-major, ld = S2_W
  T* hcol = Dw + (size_t)(p - 1) * S2_W * S2_W;         // column jc of H_1, rows lo..hi
  T* rs = hcol + S2_W;                                  // [S2_K][E]
  double* rc = reinterpret_cast<double*>(rs + (size_t)S2_K * E);
  T* H1 = cx.Hp(1);
  const int nZ = cx.wantZ ? n : 0;
  long long acc0 = 0, acc1 = 0, acc2 = 0, acc3 = 0, tq = 0;  // phase cycles (debug)
  for (int jc = 1; jc <= n - 2; jc++) {
    for (int i0 = n; i0 >= jc + 2; i0 -= S2_K) {
      const int i1 = max(jc + 2, i0 - S2_K + 1);
      const int kb = i0 - i1 + 1, W = kb + 1, lo = i1 - 1, hi = i0;  // rows / columns lo..hi (1-based)
      // (1) windows and the generating column into shared memory
      if (cx.prof) tq = clock64();
      for (int e = tid; e < (p - 1) * W * W; e += nt) {
        const int f = e / (W * W), q = e - f * W * W, r = q % W, c = q / W;
        Dw[(size_t)f * S2_W * S2_W + r + c * S2_W] = ldg_(&PSD_GE(cx.Hp(2 + f), ld, lo + r, lo + c));
      }
      for (int e = tid; e < W; e += nt) hcol[e] = ldg_(&PSD_GE(H1, ld, lo + e, jc));
      __syncthreads();
      if (cx.prof) { const long long t = clock64(); acc0 += t - tq; tq = t; }
      // (2) the kb rotation chains on the windows, as a wavefront: cell (t, f) = rotation t at
      // chain position f (f = 0: generation from column jc of H_1; f >= 1: factor l = p + 1 - f)
      // needs (t, f-1) for its incoming rotation and (t-1, f) for the state of its window, so all
      // cells of an anti-diagonal t + f = d are independent: one warp per chain position, a CTA
      // barrier per anti-diagonal, kb + p - 1 of them instead of kb * p serial cells.
      {
        const int nw = nt >> 5, k1 = 3 * (p - 1);
        for (int d = 1; d <= kb + p - 1; d++) {
          for (int f = warp; f < p; f += nw) {
            const int t = d - f;
            if (t < 1 || t > kb) continue;
            const int a = W - 1 - t;  // local index of the upper row / left column of the pair
            if (f == 0) {
              double c1;
              T s1, r1;
              givens_chain(hcol[a], hcol[a + 1], c1, s1, r1);
              __syncwarp();
              if (lane == 0) {
                hcol[a] = r1;
                hcol[a + 1] = Scalar<T>::zero();
                const int k = (t - 1) * E + k1;
                rc[k] = c1; rs[k] = s1;                // rows of H_1
                rc[k + 1] = c1; rs[k + 1] = conj_(s1);  // columns of Z_1
                if (p == 1) {
                  rc[k + 2] = c1; rs[k + 2] = conj_(s1);  // columns of H_1
                }
              }
              __syncwarp();
              continue;
            }
            const int l = p + 1 - f;
            double ci;
            T si;
            if (f == 1) {
              ci = rc[(t - 1) * E + k1];
              si = rs[(t - 1) * E + k1];
            } else {
              ci = rc[(t - 1) * E + 3 * (l + 1 - 2) + 2];
              si = conj_(rs[(t - 1) * E + 3 * (l + 1 - 2) + 2]);
            }
            T* D = Dw + (size_t)(l - 2) * S2_W * S2_W;
            RotChain<T> o;
            rot_chain_step<T>(cx.Sg(l), ci, si, D[a + a * S2_W], D[a + (a + 1) * S2_W], D[a + 1 + (a + 1) * S2_W], o);
            __syncwarp();
            if (lane < a) {  // column rotation on the window rows above the block
              T* pa = D + lane + a * S2_W;
              const T sv = conj_(o.sR), x = pa[0], y = pa[S2_W];
              pa[0] = o.cR * x + sv * y;
              pa[S2_W] = o.cR * y - conj_(sv) * x;
            } else if (lane >= a + 2 && lane < W) {  // row rotation on the window columns right of it
              T* pa = D + a + lane * S2_W;
              const T x = pa[0], y = pa[1];
              pa[0] = o.cL * x + o.sL * y;
              pa[1] = o.cL * y - conj_(o.sL) * x;
            } else if (lane == a) {
              D[a + a * S2_W] = o.m00;
              D[a + (a + 1) * S2_W] = o.m01;
              D[a + 1 + (a + 1) * S2_W] = o.m11;
              const int k = (t - 1) * E + 3 * (l - 2);
              rc[k] = o.cR; rs[k] = conj_(o.sR);
              rc[k + 1] = o.cL; rs[k + 1] = o.sL;
              rc[k + 2] = o.co; rs[k + 2] = conj_(o.so);
              if (l == 2) {
                rc[(t - 1) * E + k1 + 2] = o.co;
                rs[(t - 1) * E + k1 + 2] = conj_(o.so);  // columns of H_1
              }
            }
            __syncwarp();
          }
          __syncthreads();
        }
      }
      __syncthreads();
      if (cx.prof) { const long long t = clock64(); acc1 += t - tq; tq = t; }
      // (3) pass A: every strip outside the windows, H_1 from the left, all Z
      {
        const int nAb = lo - 1, nRt = n - hi, per = nAb + nRt + nZ, nf = (p - 1) * per;
        const int nH1 = n - jc, total = nf + nH1 + nZ;
        const float rper = per > 0 ? 1.0f / (float)per : 0.0f;
        const int k1 = 3 * (p - 1);
        for (int w = tid; w < total; w += nt) {
          T* ptr;
          long long st;
          int k;
          if (w < nf) {
            int f, r;
            split_index(w, per, rper, f, r);
            const int l = 2 + f;
            k = 3 * f;
            if (r < nAb) {
              ptr = &PSD_GE(cx.Hp(l), ld, 1 + r, lo);
              st = ld;
            } else if (r < nAb + nRt) {
              ptr = &PSD_GE(cx.Hp(l), ld, lo, hi + 1 + (r - nAb));
              st = 1;
              k += 1;
            } else {
              ptr = &PSD_GE(cx.Zp(l), ldz, 1 + (r - nAb - nRt), lo);
              st = ldz;
              k += 2;
            }
          } else {
            const int r = w - nf;
            if (r < nH1) {
              ptr = &PSD_GE(H1, ld, lo, jc + 1 + r);
              st = 1;
              k = k1;
            } else {
              ptr = &PSD_GE(cx.Zp(1), ldz, 1 + (r - nH1), lo);
              st = ldz;
              k = k1 + 1;
            }
          }
          if (kb == S2_K)
            s2_apply_seq<T, true>(ptr, st, kb, rc + k, rs + k, E);
          else
            s2_apply_seq<T, false>(ptr, st, kb, rc + k, rs + k, E);
        }
      }
      __syncthreads();
      if (cx.prof) { const long long t = clock64(); acc2 += t - tq; tq = t; }
      // (4) pass B: H_1 from the right; windows and the generating column back to global memory
      for (int r = tid; r < n; r += nt) {
        if (kb == S2_K)
          s2_apply_seq<T, true>(&PSD_GE(H1, ld, 1 + r, lo), ld, kb, rc + 3 * (p - 1) + 2, rs + 3 * (p - 1) + 2, E);
        else
          s2_apply_seq<T, false>(&PSD_GE(H1, ld, 1 + r, lo), ld, kb, rc + 3 * (p - 1) + 2, rs + 3 * (p - 1) + 2, E);
      }
      for (int e = tid; e < (p - 1) * W * W; e += nt) {
        const int f = e / (W * W), q = e - f * W * W, r = q % W, c = q / W;
        if (r <= c) stg_(&PSD_GE(cx.Hp(2 + f), ld, lo + r, lo + c), Dw[(size_t)f * S2_W * S2_W + r + c * S2_W]);
      }
      for (int e = tid; e < W; e += nt) stg_(&PSD_GE(H1, ld, lo + e, jc), hcol[e]);
      __syncthreads();
      if (cx.prof) acc3 += clock64() - tq;
    }
  }
  if (cx.prof && tid == 0 && blockIdx.x == 0)
    printf("[psd stage2 windowed] load %lld  window %lld  passA %lld  passB+store %lld cycles\n", acc0, acc1, acc2, acc3);
}

// _phessenberg!(A, S) (generalized.jl:988-1082) with the Q accumulation fused in.
template <class T>
PSD_DEV void gphessenberg_cta(const GCtx<T>& cx) {
  const int n = cx.n, p = cx.p, tid = cx.tid, nt = cx.nt, ld = cx.ldh;
  if (cx.wantZ) {
    for (int l = 1; l <= p; l++) {
      T* Zl = cx.Zp(l);
      for (int e = tid; e < n * n; e += nt) {
        const int r = e % n, c = e / n;
        Zl[r + (size_t)c * cx.ldz] = (r == c) ? Scalar<T>::one() : Scalar<T>::zero();
      }
    }
  }
  __syncthreads();
  // Stage 1 (:1009-1028)
  for (int l = p; l >= 2; l--) {
    T* Al = cx.Hp(l);
    T* Am = cx.Hp(l - 1);
    T* Ql = cx.wantZ ? cx.Zp(l) : nullptr;
    const bool sm1 = cx.Sg(l - 1);
    if (cx.blk) {
      BlkWork<T> W;
      W.Vs = cx.blk;
      W.Ts = cx.blk + (size_t)n * S1_NB;
      W.Gs = W.Ts + S1_NB * S1_NB;
      W.taus = W.Gs + S1_NB * S1_NB;
      stage1_blocked(cx, l, W);
    } else if (cx.Sg(l)) {
      for (int k = 1; k <= n - 1; k++) stage1_qr_step(cx, Al, Am, sm1, Ql, k);
    } else {
      for (int k = n; k >= 2; k--) stage1_rq_step(cx, Al, Am, sm1, Ql, k);
    }
  }
  if (cx.prof && tid == 0) cx.prof[0] = clock64();
  // Stage 2 (:1034-1079): rotation (i-1, i) zeroing A_1[i, jc], chased through all factors
  if (cx.s2ws >= 0) {
    stage2_windowed<T>(cx, cx.s2ws);
    return;
  }
  T* A1 = cx.Hp(1);
  for (int jc = 1; jc <= n - 2; jc++) {
    for (int i = n; i >= jc + 2; i--) {
      const T f = PSD_GE(A1, ld, i - 1, jc), g = PSD_GE(A1, ld, i, jc);
      if (is_zero(g)) continue;  // identity rotation (uniform over the CTA)
      double c;
      T s, r;
      givens_t(f, g, c, s, r);
      chase_rotation(cx, i - 1, c, s, jc, r, jc + 1, n, 1, n);
    }
  }
}

// x = m 2^k exactly, with the larger of |Re m|, |Im m| in [0.5, 1); m = x and k = 0 for a zero.
// Products of diagonal entries multiply (divide) mantissas and add (subtract) exponents: the raw
// product overflows above about 9e307, a quotient by a subnormal overflows, and a product with a
// subnormal rounds onto the subnormal grid.  In the normal range the result is the same, bit for bit.
PSD_DEV double pow2_split(double x, int& k) {
  k = 0;
  if (x == 0.0 || !isfinite(x)) return x;
  (void)frexp(x, &k);
  return scalbn(x, -k);
}
PSD_DEV cplx pow2_split(cplx x, int& k) {
  k = 0;
  const double big = fmax(fabs(x.x), fabs(x.y));
  if (big == 0.0 || !isfinite(big)) return x;
  (void)frexp(big, &k);
  return mk(scalbn(x.x, -k), scalbn(x.y, -k));
}

// generalized.jl:939-976 (_safeprod): x_1^{s_1} prod x_l^{s_l} = alpha / beta * 2^scale with
// |alpha| in [1,2) or 0 and beta in {0,1}.  d[l-1] = diagonal entry of factor l.  Unlike the
// reference, each x_l enters split into mantissa and exponent (pow2_split).
template <class T, class F>
PSD_DEV void safeprod(int p, const unsigned char* S, F diag_of, T& alpha, int& beta, long long& scale) {
  alpha = Scalar<T>::one();
  beta = 1;
  scale = 0;
  for (int i = 1; i <= p; i++) {
    const T xi = diag_of(i);
    int k;
    const T mi = pow2_split(xi, k);
    if (S[i - 1]) {
      alpha = alpha * mi;
      scale += k;
    } else {
      if (is_zero(xi)) {
        beta = 0;
      } else {
        alpha = alpha / mi;
        scale -= k;
      }
    }
    double aa = abs_(alpha);
    if (aa == 0.0) {
      alpha = Scalar<T>::zero();
      scale = 0;
      if (beta == 0) return;
    } else if (isfinite(aa)) {
      int e;
      (void)frexp(aa, &e);  // aa = f 2^e, f in [0.5,1)  ->  |alpha| 2^-(e-1) in [1,2)
      alpha = alpha * scalbn(1.0, -(e - 1));
      // guard against hypot rounding at the boundary
      aa = abs_(alpha);
      if (aa >= 2.0) { alpha = alpha * 0.5; e++; }
      else if (aa < 1.0) { alpha = alpha * 2.0; e--; }
      scale += (e - 1);
    }
  }
}

}  // namespace psd
