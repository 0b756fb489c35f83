// Complex (generalized) periodic Schur kernel: one CTA per periodic problem.
//
// Replaces, on device, the reference call chain
//   pschur!(A, S, lr; wantZ, wantT)          generalized.jl:108-148     (driver, :L reversal)
//   _phessenberg!(A, S)                       generalized.jl:988-1082    (psd_gen_common.cuh)
//   pschur!(H1, Hs, S; ...)  (MB03BZ-style)   generalized.jl:166-931     (cpqz_cta below)
//   _safeprod                                 generalized.jl:939-976
// and, with S = trues, the complex standard wrapper PeriodicSchurDecompositions.jl:1106-1111.
//
// Deliberate deviations from rarely taken reference branches (SURVEY.md appendix A.7):
//  * the exceptional shift uses a deterministic golden-ratio sequence instead of rand(T,2)
//    (generalized.jl:782);
//  * when Test 2 (S+ diagonal) fires, Test 3 is skipped and the controlled zero shift (Test 4)
//    only runs when neither fired, as in SLICOT MB03BZ (the Julia text lets a later test
//    overwrite ldeflate/jdeflate, :341-353).
#pragma once
#include "psd_gen_common.cuh"

namespace psd {

template <class T>
struct GpqzParams {
  int n, p;
  long long batch;
  int left, wantT, wantZ, maxitfac;
  int skip_reduce;          // input already Hessenberg-triangular (pschur!(H1,Hs,S) entry, :166)
  int reduce_only;          // stop after _phessenberg!(A, S): A <- H factors, Z <- Q (no eigenvalues)
  const unsigned char* S;   // [p] user order (device memory)
  T* A;                     // [batch][p][n*n] in/out, user order
  T* Z;                     // [batch][p][n*n] out (reference result order) or nullptr
  cplx* alpha;              // [batch][n]
  T* beta;                  // [batch][n] (complex for the complex path, real for the real one)
  long long* scale;         // [batch][n]
  int* info;                // [batch]
  int use_smem, ldh;
  int blocked_stage1;       // dynamic shared memory holds blk_work_scalars(n) more scalars after the small state
  int windowed_qz;          // dynamic shared memory also covers qzw_work_doubles(p) doubles (real path, same area)
  int windowed_stage2;      // dynamic shared memory also covers s2_work_scalars(p) scalars (same area as the blocked Stage 1)
  int deep;                 // use the deep (table-driven, single-pass) rotation chases
  int debug;                // print a phase breakdown (cycles) for the problems of CTA 0
  unsigned long long* counter;
  int* pexp = nullptr;      // [gridDim.x][p] gpschur_kernel: power-of-two exponents of the factors of the
                            // problem a CTA works on (factor_scale_exponents)
};

// doubles of per-CTA small state: Gc (n+2), Gs 2(n+2), stage (complex: 2(4+3(p-1)); real double
// chase: 9+6(p-1)), S bytes
__host__ __device__ inline long long cq_stage_doubles(int p) { return 10LL + 6 * (p > 1 ? p - 1 : 0); }
// offset of the rotation table of the deep chase variants (12 (p+1) doubles) inside `small`
__host__ __device__ inline long long cq_rots_offset(int n, int p) {
  return (5LL * (n + 2) + 2 * cq_stage_doubles(p) + (p + 15) / 8 + 2 + 1) & ~1LL;
}
__host__ __device__ inline long long cq_small_doubles(int n, int p) {
  return cq_rots_offset(n, p) + 12LL * (p + 1);
}

template <class T>
struct GqState {
  double* Gc;
  T* Gs;
  int* key;  // shared scratch for the parallel deflation scans
};

// Test 1 (generalized.jl:260-278): bottom-up scan for a negligible subdiagonal of H_1.
template <class T>
PSD_DEV bool cq_check_hess(const GCtx<T>& cx, const GqState<T>& st, int ilo, int ilast, double ulp,
                           double smlnum, int& jlo) {
  T* H1 = cx.Hp(1);
  const int ld = cx.ldh;
  if (cx.tid == 0) *st.key = 0;
  __syncthreads();
  for (int j = ilast - cx.tid; j >= ilo + 1; j -= cx.nt) {
    double tol = abs_(PSD_GE(H1, ld, j - 1, j - 1)) + abs_(PSD_GE(H1, ld, j, j));
    if (tol == 0.0) tol = g_opnorm1(H1, ld, ilo, j, ilo, j, false);
    tol = fmax(ulp * tol, smlnum);
    if (abs_(PSD_GE(H1, ld, j, j - 1)) <= tol) atomicMax(st.key, j);
  }
  __syncthreads();
  const int jf = *st.key;
  __syncthreads();
  jlo = ilo;
  if (jf > 0) {
    if (cx.team) cx.sync();  // every CTA has finished its (redundant) scan
    if (cx.lead && cx.tid == 0) PSD_GE(H1, ld, jf, jf - 1) = Scalar<T>::zero();
    jlo = jf;
    cx.sync();
    return jf == ilast;
  }
  return false;
}

// Tests 2/3 (generalized.jl:280-299, 327-353): first factor l (ascending) with signature
// `sign` that has a negligible diagonal entry in jlo..ilast, and the largest such j.
template <class T>
PSD_DEV bool cq_check_tr(const GCtx<T>& cx, const GqState<T>& st, bool sign, int jlo, int ilast,
                         double ulp, double smlnum, int& ldef, int& jdef) {
  const int n = cx.n, p = cx.p, ld = cx.ldh;
  if (cx.tid == 0) *st.key = 0;
  __syncthreads();
  const int span = ilast - jlo + 1;
  for (int w = cx.tid; w < (p - 1) * span; w += cx.nt) {
    const int l = 2 + w / span, j = jlo + w % span;
    if (cx.Sg(l) != sign) continue;
    const T* Hl = cx.Hp(l);
    double tol;
    if (j == ilast)
      tol = abs_(PSD_GE(Hl, ld, j - 1, j));
    else if (j == jlo)
      tol = abs_(PSD_GE(Hl, ld, j, j + 1));
    else
      tol = abs_(PSD_GE(Hl, ld, j - 1, j)) + abs_(PSD_GE(Hl, ld, j, j + 1));
    if (tol == 0.0) tol = g_opnorm1(Hl, ld, jlo, j, jlo, j, true);
    tol = fmax(ulp * tol, smlnum);
    if (abs_(PSD_GE(Hl, ld, j, j)) <= tol) atomicMax(st.key, (p + 1 - l) * (n + 1) + j);
  }
  __syncthreads();
  const int k = *st.key;
  __syncthreads();
  if (k == 0) return false;
  ldef = p + 1 - k / (n + 1);
  jdef = k % (n + 1);
  if (cx.team) cx.sync();
  if (cx.lead && cx.tid == 0) PSD_GE(cx.Hp(ldef), ld, jdef, jdef) = Scalar<T>::zero();
  cx.sync();
  return true;
}

// rmul!(M, G_j') for j = j0, j0+dj, ..., j1 in sequence, G_j = Givens(j+oa, j+ob, Gc[j], Gs[j]),
// all rows: one thread per row, no barrier inside.
template <class T>
PSD_DEV void cq_rmul_seq(const GCtx<T>& cx, const GqState<T>& st, T* M, int ld, int j0, int j1,
                         int dj, int oa, int ob) {
  for (int row = 1 + cx.wtid; row <= cx.n; row += cx.wnt)
    for (int j = j0; dj > 0 ? j <= j1 : j >= j1; j += dj)
      rot_pair_cols(M, ld, j + oa, j + ob, row, st.Gc[j], st.Gs[j]);
  cx.sync();
}

#define CQ_SETG(j, c, s)    \
  do {                      \
    if (cx.tid == 0) {      \
      st.Gc[j] = (c);       \
      st.Gs[j] = (s);       \
    }                       \
  } while (0)

// ==========================================================================================
// Real path (rgeneralized.jl:655-1054): double-shift sweeps with two rotations per step and
// 2x2 block handling.
//
// How this differs from the reference text (results agree to the tolerances of BASELINE.json;
// shifts only steer convergence):
//  * the two starting rotations come from the first column of the double-shift polynomial of the
//    product H_1 T, T = prod_{l>=2} H_l^{s_l}, evaluated from the leading and trailing 3x3 blocks
//    of the triangular factors with a running power-of-two scale (what the real standard path
//    does with its product band, PeriodicSchurDecompositions.jl:474-529, 730-803) instead of
//    MB03AF's implicit rotation chains (_qzrots, :1140-1359); the reference's explicit-shift
//    branch (:804-887) is not replicated (it reads undefined names, SURVEY.md appendix A.7);
//    every 10th iteration on a block takes a deterministic exceptional shift vector;
//  * the sweep always enters at Z_1 (rows of H_1), which the reference does only for p == 1
//    (:944-950); for p > 1 it enters between H_1 and H_2 (:890-943) - the same similarity of a
//    cyclic shift of the product;
//  * a 2x2 block is classified by dlanv2 (gs2x2, rschur2x2.jl:9-96) on the explicitly formed,
//    scaled 2x2 product; a real pair is split by chasing dlanv2's rotation through the factors
//    (the role of _rp2x2ssr! + the "perfect shift" chain, :685-745), repeated by the outer loop
//    until Test 1 deflates; a complex pair is left unstandardised in T_1 as in the reference
//    (:748-790) with alpha, beta, alphascale taken from the scaled product.
// ==========================================================================================

// (a1, a2) <- [c s; -s c] (a1, a2): the same formula serves lmul!(G, .) on a row pair and
// rmul!(., G') on a column pair for real data.
PSD_DEV void rrot(double& a1, double& a2, double c, double s) {
  const double t = c * a1 + s * a2;
  a2 = c * a2 - s * a1;
  a1 = t;
}
struct Rot2 {
  double c1, s1;  // G2 = Givens(j, j+1)
  double c2, s2;  // G1 = Givens(j+1, j+2), applied first
};
PSD_DEV void rot3(double& a0, double& a1, double& a2, const Rot2& g) {
  rrot(a1, a2, g.c2, g.s2);
  rrot(a0, a1, g.c1, g.s1);
}

// Independent 3-element items (a[0], a[st], a[2 st]) <- rot3(., g[sel]); BULK_U of them are loaded
// before any is stored (memory-latency bound at the larger sizes, see bulk_rot2).
template <class Item>
PSD_DEV void bulk_rot3(int tid, int nt, int total, const Rot2 (&g)[3], Item&& item) {
  for (int w0 = tid; w0 < total; w0 += BULK_U * nt) {
    double* pa[BULK_U];
    long long st[BULK_U];
    int sel[BULK_U];
    double v0[BULK_U], v1[BULK_U], v2[BULK_U];
#pragma unroll
    for (int u = 0; u < BULK_U; u++) {
      const int w = w0 + u * nt;
      pa[u] = nullptr;
      if (w < total) item(w, pa[u], st[u], sel[u]);
    }
#pragma unroll
    for (int u = 0; u < BULK_U; u++)
      if (pa[u]) {
        v0[u] = pa[u][0];
        v1[u] = pa[u][st[u]];
        v2[u] = pa[u][2 * st[u]];
      }
#pragma unroll
    for (int u = 0; u < BULK_U; u++)
      if (pa[u]) {
        const Rot2 gg = (sel[u] == 0) ? g[0] : (sel[u] == 1) ? g[1] : g[2];
        rot3(v0[u], v1[u], v2[u], gg);
        pa[u][0] = v0[u];
        pa[u][st[u]] = v1[u];
        pa[u][2 * st[u]] = v2[u];
      }
  }
}

// Deep variant of bulk_rot3 (see bulk_rot2_tab): the rotation pair of item w is entry k of a
// shared-memory table covering all factors of one chase.  item(w, a, st, k).
template <int U, class Item>
PSD_DEV void bulk_rot3_tab(int tid, int nt, int total, const Rot2* tab, Item&& item) {
  for (int w0 = tid; w0 < total; w0 += U * nt) {
    double* pa[U];
    int st[U], kk[U];
    double v0[U], v1[U], v2[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int w = w0 + u * nt;
      pa[u] = nullptr;
      if (w < total) item(w, pa[u], st[u], kk[u]);
    }
#pragma unroll
    for (int u = 0; u < U; u++)
      if (pa[u]) {
        v0[u] = pa[u][0];
        v1[u] = pa[u][st[u]];
        v2[u] = pa[u][2 * st[u]];
      }
#pragma unroll
    for (int u = 0; u < U; u++)
      if (pa[u]) {
        const Rot2 gg = tab[kk[u]];
        rot3(v0[u], v1[u], v2[u], gg);
        pa[u][0] = v0[u];
        pa[u][st[u]] = v1[u];
        pa[u][2 * st[u]] = v2[u];
      }
  }
}

// One link of the double-rotation chain through the 3x3 diagonal block B (upper triangular,
// B = {b00 b01 b02 b11 b12 b22}) of a triangular factor; gout travels on, B is updated in place.
PSD_DEV void rot2_chain_step(bool sl, const Rot2& gin, double (&B)[6], Rot2& gout) {
  double &B00 = B[0], &B01 = B[1], &B02 = B[2], &B11 = B[3], &B12 = B[4], &B22 = B[5];
  double B10 = 0.0, B21 = 0.0, r;
  if (sl) {
    // columns (j+1,j+2) <- G1in; rows (j+1,j+2) re-triangularised by G1out;
    // columns (j,j+1) <- G2in; rows (j,j+1) re-triangularised by G2out   (:980-991)
    rrot(B01, B02, gin.c2, gin.s2);
    rrot(B11, B12, gin.c2, gin.s2);
    rrot(B21, B22, gin.c2, gin.s2);
    givens_chain(B11, B21, gout.c2, gout.s2, r);
    B11 = r; B21 = 0.0;
    rrot(B12, B22, gout.c2, gout.s2);
    rrot(B00, B01, gin.c1, gin.s1);
    rrot(B10, B11, gin.c1, gin.s1);
    givens_chain(B00, B10, gout.c1, gout.s1, r);
    B00 = r; B10 = 0.0;
    rrot(B01, B11, gout.c1, gout.s1);
    rrot(B02, B12, gout.c1, gout.s1);
  } else {
    // rows (j+1,j+2) <- G1in; columns (j+1,j+2) by G1out (rows <= j+1);
    // rows (j,j+1) <- G2in; columns (j,j+1) by G2out (rows <= j)           (:993-1004)
    rrot(B11, B21, gin.c2, gin.s2);
    rrot(B12, B22, gin.c2, gin.s2);
    givens_chain(B22, -B21, gout.c2, gout.s2, r);
    B22 = r; B21 = 0.0;
    rrot(B01, B02, gout.c2, gout.s2);
    rrot(B11, B12, gout.c2, gout.s2);
    rrot(B00, B10, gin.c1, gin.s1);
    rrot(B01, B11, gin.c1, gin.s1);
    rrot(B02, B12, gin.c1, gin.s1);
    givens_chain(B11, -B10, gout.c1, gout.s1, r);
    B11 = r; B10 = 0.0;
    rrot(B00, B01, gout.c1, gout.s1);
  }
}

// chase_double: the two rotations G1 = Givens(j+1,j+2), G2 = Givens(j,j+1) act on rows j..j+2
// of H_1 (columns j..clast), are propagated through factors p..2 (rgeneralized.jl:977-1010) and
// return to columns j..j+2 of H_1 (rows rfirst..h1r1).  Same organisation as chase_rotation:
// the 3x3 diagonal blocks are processed in registers by every thread, bulk updates touch
// disjoint memory, blocks are staged in shared memory and written back between two barriers.
__device__ __noinline__ void chase_double(const GCtx<double>& cx, int j, Rot2 gin, int zcol, double r1, int clast,
                          int rfirst, int h1r1) {
  const int n = cx.n, p = cx.p, tid = cx.tid, nt = cx.nt, ld = cx.ldh;
  double* H1 = cx.Hp(1);
  // one parallel load of every 3x3 diagonal block (H_1: 9 entries, factor l: 6 at 9+6(l-2))
  {
    double* in = cx.stage_in;
    for (int e = tid; e < 9 + 6 * (p - 1); e += nt) {
      if (e < 9) {
        in[e] = PSD_GE(H1, ld, j + e / 3, j + e % 3);
      } else {
        const int l = 2 + (e - 9) / 6, w = (e - 9) % 6;
        const int rr = (w < 3) ? 0 : (w < 5) ? 1 : 2;
        const int cc = (w < 3) ? w : (w < 5) ? (w - 2) : 2;
        in[e] = PSD_GE(cx.Hp(l), ld, j + rr, j + cc);
      }
    }
    __syncthreads();
  }
  const double* bin = cx.stage_in;
  double X[3][3];
#pragma unroll
  for (int r = 0; r < 3; r++)
#pragma unroll
    for (int c = 0; c < 3; c++) X[r][c] = bin[3 * r + c];
  const Rot2 g0 = gin;
  if (cx.rots) {
    // Deep variant (see chase_rotation): chain first, then one bulk pass over all factors.
    Rot2* tab = reinterpret_cast<Rot2*>(cx.rots);
    const int k1 = 3 * (p - 1);
    if (tid == 0) {
      for (int l = p; l >= 2; l--) {
        const double* bl = bin + 9 + 6 * (l - 2);
        double Bk[6] = {bl[0], bl[1], bl[2], bl[3], bl[4], bl[5]};
        Rot2 gout;
        const bool sl = cx.Sg(l);
        rot2_chain_step(sl, gin, Bk, gout);
        const int k = 3 * (l - 2);
        tab[k] = sl ? gin : gout;      // columns (rows above the block)
        tab[k + 1] = sl ? gout : gin;  // rows (columns right of the block)
        tab[k + 2] = gout;             // Z_l
        double* sg = cx.stage + 9 + 6 * (l - 2);
#pragma unroll
        for (int e = 0; e < 6; e++) sg[e] = Bk[e];
        gin = gout;
      }
      tab[k1] = g0;       // rows of H_1 and columns of Z_1
      tab[k1 + 1] = gin;  // columns of H_1
#pragma unroll
      for (int c = 0; c < 3; c++) rot3(X[0][c], X[1][c], X[2][c], g0);
#pragma unroll
      for (int r = 0; r < 3; r++) rot3(X[r][0], X[r][1], X[r][2], gin);
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) cx.stage[3 * r + c] = X[r][c];
    }
    __syncthreads();
    const int nR = j - rfirst, nL = clast - (j + 2), nZ = cx.wantZ ? n : 0;
    const int per = nR + nL + nZ, nf = (p - 1) * per;
    const int nR1 = (h1r1 - rfirst + 1) - 3;
    const int total = nf + nL + nZ + nR1;
    const float rper = per > 0 ? 1.0f / (float)per : 0.0f;
    const int ldz = cx.ldz;
    auto deep_item = [&](int w, double*& a, int& st, int& k) {
      if (w < nf) {
        int f, r;
        split_index(w, per, rper, f, r);
        const int l = 2 + f;
        k = 3 * f;
        if (r < nR) {
          a = &PSD_GE(cx.Hp(l), ld, rfirst + r, j);
          st = ld;
        } else if (r < nR + nL) {
          a = &PSD_GE(cx.Hp(l), ld, j, j + 3 + (r - nR));
          st = 1;
          k += 1;
        } else {
          a = &PSD_GE(cx.Zp(l), ldz, 1 + (r - nR - nL), j);
          st = ldz;
          k += 2;
        }
      } else {
        int r = w - nf;
        if (r < nL) {
          a = &PSD_GE(H1, ld, j, j + 3 + r);
          st = 1;
          k = k1;
        } else if (r < nL + nZ) {
          a = &PSD_GE(cx.Zp(1), ldz, 1 + (r - nL), j);
          st = ldz;
          k = k1;
        } else {
          int row = rfirst + (r - nL - nZ);
          if (row >= j) row += 3;
          a = &PSD_GE(H1, ld, row, j);
          st = ld;
          k = k1 + 1;
        }
      }
    };
    if (cx.deep_u == 8)
      bulk_rot3_tab<6>(cx.wtid, cx.wnt, total, tab, deep_item);
    else if (cx.deep_u == 2)
      bulk_rot3_tab<2>(cx.wtid, cx.wnt, total, tab, deep_item);
    else
      bulk_rot3_tab<4>(cx.wtid, cx.wnt, total, tab, deep_item);
    cx.sync();
    for (int l = 1 + tid; cx.lead && l <= p; l += nt) {
      if (l == 1) {
        for (int r = 0; r < 3; r++)
          for (int c = 0; c < 3; c++) PSD_GE(H1, ld, j + r, j + c) = cx.stage[3 * r + c];
        if (zcol > 0) {
          PSD_GE(H1, ld, j, zcol) = r1;
          PSD_GE(H1, ld, j + 1, zcol) = 0.0;
          PSD_GE(H1, ld, j + 2, zcol) = 0.0;
        }
      } else {
        double* Hl = cx.Hp(l);
        const double* sg = cx.stage + 9 + 6 * (l - 2);
        PSD_GE(Hl, ld, j, j) = sg[0]; PSD_GE(Hl, ld, j, j + 1) = sg[1]; PSD_GE(Hl, ld, j, j + 2) = sg[2];
        PSD_GE(Hl, ld, j + 1, j) = 0.0; PSD_GE(Hl, ld, j + 1, j + 1) = sg[3]; PSD_GE(Hl, ld, j + 1, j + 2) = sg[4];
        PSD_GE(Hl, ld, j + 2, j) = 0.0; PSD_GE(Hl, ld, j + 2, j + 1) = 0.0; PSD_GE(Hl, ld, j + 2, j + 2) = sg[5];
      }
    }
    cx.sync();
    return;
  }
  {  // left-only columns of H_1 and Z_1
    const int nL = clast - (j + 2);
    const int nZ = cx.wantZ ? n : 0;
    double* Z1 = cx.wantZ ? cx.Zp(1) : nullptr;
    const Rot2 gs[3] = {g0, g0, g0};
    const int ldz = cx.ldz;
    bulk_rot3(cx.wtid, cx.wnt, nL + nZ, gs, [&](int w, double*& a, long long& st, int& sel) {
      sel = 0;
      if (w < nL) {
        a = &PSD_GE(H1, ld, j, j + 3 + w);
        st = 1;
      } else {
        a = &PSD_GE(Z1, ldz, 1 + (w - nL), j);
        st = ldz;
      }
    });
  }
  for (int l = p; l >= 2; l--) {
    double* Hl = cx.Hp(l);
    const double* bl = bin + 9 + 6 * (l - 2);
    double Bk[6] = {bl[0], bl[1], bl[2], bl[3], bl[4], bl[5]};
    Rot2 gout;
    const bool sl = cx.Sg(l);
    rot2_chain_step(sl, gin, Bk, gout);
    {
      const Rot2 gR = sl ? gin : gout;  // acts on columns (rows above the block)
      const Rot2 gL = sl ? gout : gin;  // acts on rows (columns right of the block)
      const int nR = j - rfirst, nL = clast - (j + 2);
      const int nZ = cx.wantZ ? n : 0;
      double* Zl = cx.wantZ ? cx.Zp(l) : nullptr;
      const Rot2 gs[3] = {gR, gL, gout};
      const int ldz = cx.ldz;
      bulk_rot3(cx.wtid, cx.wnt, nR + nL + nZ, gs, [&](int w, double*& a, long long& st, int& sel) {
        if (w < nR) {
          a = &PSD_GE(Hl, ld, rfirst + w, j);
          st = ld;
          sel = 0;
        } else if (w < nR + nL) {
          a = &PSD_GE(Hl, ld, j, j + 3 + (w - nR));
          st = 1;
          sel = 1;
        } else {
          a = &PSD_GE(Zl, ldz, 1 + (w - nR - nL), j);
          st = ldz;
          sel = 2;
        }
      });
      if (tid == 0) {
        double* sg = cx.stage + 9 + 6 * (l - 2);
        sg[0] = Bk[0]; sg[1] = Bk[1]; sg[2] = Bk[2]; sg[3] = Bk[3]; sg[4] = Bk[4]; sg[5] = Bk[5];
      }
    }
    gin = gout;
  }
  {  // right-only rows of H_1 and its 3x3 overlap block
    const int nR = (h1r1 - rfirst + 1) - 3;
    const Rot2 gs[3] = {gin, gin, gin};
    bulk_rot3(cx.wtid, cx.wnt, nR, gs, [&](int w, double*& a, long long& st, int& sel) {
      int row = rfirst + w;
      if (row >= j) row += 3;
      a = &PSD_GE(H1, ld, row, j);
      st = ld;
      sel = 0;
    });
    if (tid == 0) {
#pragma unroll
      for (int c = 0; c < 3; c++) rot3(X[0][c], X[1][c], X[2][c], g0);
#pragma unroll
      for (int r = 0; r < 3; r++) rot3(X[r][0], X[r][1], X[r][2], gin);
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) cx.stage[3 * r + c] = X[r][c];
    }
  }
  cx.sync();
  for (int l = 1 + tid; cx.lead && l <= p; l += nt) {
    if (l == 1) {
      for (int r = 0; r < 3; r++)
        for (int c = 0; c < 3; c++) PSD_GE(H1, ld, j + r, j + c) = cx.stage[3 * r + c];
      if (zcol > 0) {
        PSD_GE(H1, ld, j, zcol) = r1;
        PSD_GE(H1, ld, j + 1, zcol) = 0.0;
        PSD_GE(H1, ld, j + 2, zcol) = 0.0;
      }
    } else {
      double* Hl = cx.Hp(l);
      const double* sg = cx.stage + 9 + 6 * (l - 2);
      PSD_GE(Hl, ld, j, j) = sg[0]; PSD_GE(Hl, ld, j, j + 1) = sg[1]; PSD_GE(Hl, ld, j, j + 2) = sg[2];
      PSD_GE(Hl, ld, j + 1, j) = 0.0; PSD_GE(Hl, ld, j + 1, j + 1) = sg[3]; PSD_GE(Hl, ld, j + 1, j + 2) = sg[4];
      PSD_GE(Hl, ld, j + 2, j) = 0.0; PSD_GE(Hl, ld, j + 2, j + 1) = 0.0; PSD_GE(Hl, ld, j + 2, j + 2) = sg[5];
    }
  }
  cx.sync();
}

// Scaled product of the KxK (K = 2 or 3) diagonal blocks at rows/cols i0..i0+K-1 of the
// triangular factors: Tm 2^e = prod_{l=2..p} H_l[blk]^{s_l} (upper triangular).  A zero
// diagonal of an inverted factor gives sing = true.  A direct block enters as U 2^ku with the largest
// entry of U in [0.5, 1); an inverted one entry by entry, split into mantissa and exponent (all
// exact), so that subnormal or near-overflow entries neither overflow nor lose bits; in the normal
// range the result is the same, bit for bit.
constexpr int kNoExp = -(1 << 30);  // exponent of a zero entry

template <int K>
PSD_DEV void tri_block_product(const GCtx<double>& cx, int i0, double (&Tm)[K][K], int& e, bool& sing) {
  const int p = cx.p, ld = cx.ldh;
#pragma unroll
  for (int r = 0; r < K; r++)
#pragma unroll
    for (int c = 0; c < K; c++) Tm[r][c] = (r == c) ? 1.0 : 0.0;
  e = 0;
  sing = false;
  for (int l = 2; l <= p; l++) {
    const double* Hl = cx.Hp(l);
    double U[K][K];
#pragma unroll
    for (int r = 0; r < K; r++)
#pragma unroll
      for (int c = 0; c < K; c++) U[r][c] = (c >= r) ? PSD_GE(Hl, ld, i0 + r, i0 + c) : 0.0;
    double N[K][K];
    if (cx.Sg(l)) {
      double mu = 0.0;
#pragma unroll
      for (int r = 0; r < K; r++)
#pragma unroll
        for (int c = 0; c < K; c++) mu = fmax(mu, fabs(U[r][c]));
      int ku = 0;
      if (mu > 0.0 && isfinite(mu)) (void)frexp(mu, &ku);
#pragma unroll
      for (int r = 0; r < K; r++)
#pragma unroll
        for (int c = 0; c < K; c++) U[r][c] = scalbn(U[r][c], -ku);
      e += ku;
      // N = Tm * U
#pragma unroll
      for (int r = 0; r < K; r++)
#pragma unroll
        for (int c = 0; c < K; c++) {
          double acc = 0.0;
#pragma unroll
          for (int k = 0; k < K; k++)
            if (k >= r && k <= c) acc = fma(Tm[r][k], U[k][c], acc);
          N[r][c] = acc;
        }
    } else {
      // N = Tm * inv(U): solve N U = Tm row by row (forward substitution over columns), with one
      // exponent per entry, N = q 2^x: a quotient by a diagonal entry far below the rest of the block
      // (a subnormal one) leaves the double range before the block is rescaled.  Each entry's terms
      // are summed at the exponent of the largest; every division is by a mantissa (pow2_split).
      double q[K][K];
      int x[K][K];
      int ex = kNoExp;
#pragma unroll
      for (int r = 0; r < K; r++)
#pragma unroll
        for (int c = 0; c < K; c++) {
          q[r][c] = 0.0;
          x[r][c] = 0;
          if (c < r) continue;
          int xm = (Tm[r][c] != 0.0) ? 0 : kNoExp;
          double um[K];
          int ue[K];
#pragma unroll
          for (int k = 0; k < K; k++) {
            um[k] = pow2_split(U[k][c], ue[k]);
            if (k >= r && k < c && q[r][k] != 0.0 && U[k][c] != 0.0) xm = max(xm, x[r][k] + ue[k]);
          }
          if (xm == kNoExp) xm = 0;
          double acc = scalbn(Tm[r][c], -xm);
#pragma unroll
          for (int k = 0; k < K; k++)
            if (k >= r && k < c)  // (a zero term keeps its sign but not its exponent, which can be huge)
              acc = fma(-q[r][k], scalbn(um[k], (q[r][k] != 0.0 && um[k] != 0.0) ? x[r][k] + ue[k] - xm : 0), acc);
          if (U[c][c] == 0.0) {
            sing = true;
            q[r][c] = acc;
            x[r][c] = xm;
          } else {
            int kd;
            const double md = pow2_split(U[c][c], kd);
            q[r][c] = acc / md;
            x[r][c] = xm - kd;
          }
          if (q[r][c] != 0.0 && isfinite(q[r][c])) {
            int eq;
            (void)frexp(q[r][c], &eq);
            ex = max(ex, eq + x[r][c]);
          }
        }
      if (ex == kNoExp) ex = 0;
#pragma unroll
      for (int r = 0; r < K; r++)
#pragma unroll
        for (int c = 0; c < K; c++) Tm[r][c] = scalbn(q[r][c], x[r][c] - ex);
      e += ex;
      continue;
    }
    double m = 0.0;
#pragma unroll
    for (int r = 0; r < K; r++)
#pragma unroll
      for (int c = 0; c < K; c++) m = fmax(m, fabs(N[r][c]));
    int ex = 0;
    if (m > 0.0 && isfinite(m)) (void)frexp(m, &ex);
    const double sc = scalbn(1.0, -ex);
#pragma unroll
    for (int r = 0; r < K; r++)
#pragma unroll
      for (int c = 0; c < K; c++) Tm[r][c] = N[r][c] * sc;
    e += ex;
  }
}

// 2x2 active block at rows j, j+1 (j = ifirst).  Returns true when the block has been split off
// as a complex pair (eigenvalues written); false after a rotation chain that drives
// H_1[j+1,j] towards zero (real pair).  `force`: accept the block as it stands.
PSD_DEV bool rq_block2x2(const GCtx<double>& cx, int j, int ifirstm, int ilastm, bool force, cplx* alpha,
                         double* beta, long long* scale) {
  const int ld = cx.ldh;
  double* H1 = cx.Hp(1);
  double Tm[2][2];
  int e;
  bool sing;
  tri_block_product<2>(cx, j, Tm, e, sing);
  const double h11 = PSD_GE(H1, ld, j, j), h12 = PSD_GE(H1, ld, j, j + 1);
  const double h21 = PSD_GE(H1, ld, j + 1, j), h22 = PSD_GE(H1, ld, j + 1, j + 1);
  // M = H1blk * Tm (Tm upper triangular)
  double a = h11 * Tm[0][0], b = fma(h11, Tm[0][1], h12 * Tm[1][1]);
  double c = h21 * Tm[0][0], d = fma(h21, Tm[0][1], h22 * Tm[1][1]);
  double cs, sn, w1r, w1i, w2r, w2i;
  gs2x2(a, b, c, d, cs, sn, w1r, w1i, w2r, w2i);
  if (w1i == 0.0 && !force) {
    // real pair: rotate rows j, j+1 of H_1 by dlanv2's rotation and chase it round the cycle
    chase_rotation<double>(cx, j, cs, sn, 0, 0.0, j, ilastm, ifirstm, min(j + 2, ilastm));
    return false;
  }
  cx.sync();
  if (cx.lead && cx.tid == 0) {
    const double lr[2] = {w1r, w2r}, li[2] = {w1i, w2i};
    for (int k = 0; k < 2; k++) {
      const double m = hypot(lr[k], li[k]);
      if (m == 0.0 || !isfinite(m)) {
        alpha[j - 1 + k] = mk(lr[k], li[k]);
        scale[j - 1 + k] = 0;
      } else {
        int ex;
        (void)frexp(m, &ex);
        const double sc = scalbn(1.0, -(ex - 1));
        alpha[j - 1 + k] = mk(lr[k] * sc, li[k] * sc);
        scale[j - 1 + k] = (long long)e + (ex - 1);
      }
      beta[j - 1 + k] = sing ? 0.0 : 1.0;
    }
    if (w1i == 0.0) PSD_GE(H1, ld, j + 1, j) = 0.0;  // forced acceptance of a real pair
  }
  cx.sync();
  return true;
}

// ------------------------------------------------------------------------------------------
// Windowed double-shift sweep (factors in global memory), the QZ counterpart of stage2_windowed.
//
// S3_K consecutive bulge steps j = j0 .. j0+kb-1 only read and write, as far as the rotation
// chains are concerned, the diagonal windows [j0-1, j0+kb+2]^2 of H_1 and of the triangular
// factors.  One warp runs the kb steps on copies of the windows in shared memory (bulge column,
// 3x3 blocks, in-window row / column updates) and tabulates every rotation pair; afterwards each
// thread takes one row above the windows, one column right of them or one row of a Z_l, loads its
// <= S3_W entries, applies the whole sequence of 3-element rotations in registers and stores them.
// Local index q <-> global index j0 - 1 + q; step s acts on q = s+1, s+2, s+3.
// ------------------------------------------------------------------------------------------
// S3_K = 12 steps per batch with one CTA per problem (two problems per SM share the shared
// memory); team mode uses the same (28 was measured: no gain, the serial chain dominates).
constexpr int S3_K_CTA = 12, S3_K_TEAM = 12;
__host__ __device__ inline long long qzw_work_doubles(int p, int K) {
  return (long long)p * (K + 4) * (K + 4) + 4LL * K * (3 * (p - 1) + 2) + 8;
}

template <int S3_K, bool FULL>
PSD_DEV void s3_apply_seq(double* ptr, long long stride, int qmin, int qmax, int kb, const Rot2* tab, int E) {
  constexpr int S3_W = S3_K + 4;
  double x[S3_W];
  if (FULL) {
#pragma unroll
    for (int q = 0; q < S3_W; q++) x[q] = ldg_(ptr + (long long)q * stride);
#pragma unroll
    for (int sx = 0; sx < S3_K; sx++) {
      const Rot2 g = tab[sx * E];
      rot3(x[sx + 1], x[sx + 2], x[sx + 3], g);
    }
#pragma unroll
    for (int q = 0; q < S3_W; q++) stg_(ptr + (long long)q * stride, x[q]);
    return;
  }
#pragma unroll
  for (int q = 0; q < S3_W; q++)
    if (q >= qmin && q <= qmax) x[q] = ldg_(ptr + (long long)q * stride);
#pragma unroll
  for (int sx = 0; sx < S3_K; sx++)
    if (sx < kb) {
      const Rot2 g = tab[sx * E];
      rot3(x[sx + 1], x[sx + 2], x[sx + 3], g);
    }
#pragma unroll
  for (int q = 0; q < S3_W; q++)
    if (q >= qmin && q <= qmax) stg_(ptr + (long long)q * stride, x[q]);
}

// Steps j = ifirst .. ilast-2 of one sweep; g = the two starting rotations.  The trailing single
// rotation is left to the caller.
template <int S3_K>
PSD_DEV void sweep_windowed(const GCtx<double>& cx, int ifirst, int ilast, int ifirstm, int ilastm, Rot2 g,
                            long long ws_off) {
  const int n = cx.n, p = cx.p, tid = cx.tid, nt = cx.nt, ld = cx.ldh, ldz = cx.ldz;
  const int lane = tid & 31, warp = tid >> 5;
  const int E = 3 * (p - 1) + 2;
  constexpr int S3_W = S3_K + 4, WW = S3_W * S3_W;
  double* Xw = psd_smem_cq + ws_off;  // window of H_1, column-major, ld = S3_W
  double* Dw = Xw + WW;               // windows of factors 2..p
  Rot2* tab = reinterpret_cast<Rot2*>(Dw + (size_t)(p - 1) * WW);
  double* H1 = cx.Hp(1);
  const int nZ = cx.wantZ ? n : 0;
  for (int j0 = ifirst; j0 <= ilast - 2; j0 += S3_K) {
    const int j1 = min(ilast - 2, j0 + S3_K - 1), kb = j1 - j0 + 1;
    const int base = j0 - 1;  // global index of local q = 0
    const int qmin = (base >= ifirstm) ? 0 : 1;
    const int qmax = min(j1 + 3, ilast) - base;
    // (1) windows into shared memory (entries outside [qmin, qmax] are never touched)
    for (int e = tid; e < p * WW; e += nt) {
      const int f = e / WW, q = e - f * WW, r = q % S3_W, c = q / S3_W;
      if (r >= qmin && r <= qmax && c >= qmin && c <= qmax)
        (f == 0 ? Xw : Dw + (size_t)(f - 1) * WW)[r + c * S3_W] = ldg_(&PSD_GE(cx.Hp(1 + f), ld, base + r, base + c));
    }
    __syncthreads();
    // (2) one warp runs the kb bulge steps on the windows
    if (warp == 0) {
      for (int sx = 0; sx < kb; sx++) {
        const int j = j0 + sx, a = sx + 1;
        if (j > ifirst) {
          double r2, r1;
          givens_chain(Xw[a + 1 + (a - 1) * S3_W], Xw[a + 2 + (a - 1) * S3_W], g.c2, g.s2, r2);
          givens_chain(Xw[a + (a - 1) * S3_W], r2, g.c1, g.s1, r1);
          __syncwarp();
          if (lane == 0) {
            Xw[a + (a - 1) * S3_W] = r1;
            Xw[a + 1 + (a - 1) * S3_W] = 0.0;
            Xw[a + 2 + (a - 1) * S3_W] = 0.0;
          }
        }
        // rows a..a+2 of the H_1 window, columns a..qmax
        if (lane >= a && lane <= qmax) {
          double* c0 = Xw + a + lane * S3_W;
          rot3(c0[0], c0[1], c0[2], g);
        }
        if (lane == 0) tab[sx * E + 3 * (p - 1)] = g;
        Rot2 gin = g;
        for (int l = p; l >= 2; l--) {
          double* D = Dw + (size_t)(l - 2) * WW;
          double Bk[6] = {D[a + a * S3_W], D[a + (a + 1) * S3_W], D[a + (a + 2) * S3_W],
                          D[a + 1 + (a + 1) * S3_W], D[a + 1 + (a + 2) * S3_W], D[a + 2 + (a + 2) * S3_W]};
          Rot2 gout;
          const bool sl = cx.Sg(l);
          rot2_chain_step(sl, gin, Bk, gout);
          __syncwarp();
          const Rot2 gR = sl ? gin : gout, gL = sl ? gout : gin;
          if (lane >= qmin && lane < a) {  // rows above the block: columns a..a+2
            double* r0 = D + lane + a * S3_W;
            rot3(r0[0], r0[S3_W], r0[2 * S3_W], gR);
          } else if (lane >= a + 3 && lane <= qmax) {  // columns right of the block: rows a..a+2
            double* c0 = D + a + lane * S3_W;
            rot3(c0[0], c0[1], c0[2], gL);
          } else if (lane == a) {
            D[a + a * S3_W] = Bk[0]; D[a + (a + 1) * S3_W] = Bk[1]; D[a + (a + 2) * S3_W] = Bk[2];
            D[a + 1 + (a + 1) * S3_W] = Bk[3]; D[a + 1 + (a + 2) * S3_W] = Bk[4];
            D[a + 2 + (a + 2) * S3_W] = Bk[5];
            const int k = sx * E + 3 * (l - 2);
            tab[k] = gR;
            tab[k + 1] = gL;
            tab[k + 2] = gout;
          }
          __syncwarp();
          gin = gout;
        }
        __syncwarp();
        // columns a..a+2 of the H_1 window, rows qmin..min(a+3, qmax)
        if (lane >= qmin && lane <= min(a + 3, qmax)) {
          double* r0 = Xw + lane + a * S3_W;
          rot3(r0[0], r0[S3_W], r0[2 * S3_W], gin);
        }
        if (lane == 0) tab[sx * E + 3 * (p - 1) + 1] = gin;
        __syncwarp();
      }
    }
    __syncthreads();
    // (3) the strips outside the windows and all Z
    {
      const int lo = base + qmin, hi = base + qmax;
      const int nAb = lo - ifirstm, nRt = ilastm - hi, per = nAb + nRt + nZ, total = p * per;
      const float rper = per > 0 ? 1.0f / (float)per : 0.0f;
      const bool full = (qmin == 0 && qmax == S3_W - 1 && kb == S3_K);
      for (int w = cx.wtid; w < total; w += cx.wnt) {
        int f, r;
        split_index(w, per, rper, f, r);  // f = 0: H_1 / Z_1, f >= 1: factor 1 + f
        double* ptr;
        long long st;
        int k;
        if (r < nAb) {  // row above the window, window columns: column rotations
          ptr = &PSD_GE(cx.Hp(1 + f), ld, ifirstm + r, base);
          st = ld;
          k = (f == 0) ? 3 * (p - 1) + 1 : 3 * (f - 1);
        } else if (r < nAb + nRt) {  // column right of the window, window rows: row rotations
          ptr = &PSD_GE(cx.Hp(1 + f), ld, base, hi + 1 + (r - nAb));
          st = 1;
          k = (f == 0) ? 3 * (p - 1) : 3 * (f - 1) + 1;
        } else {
          ptr = &PSD_GE(cx.Zp(1 + f), ldz, 1 + (r - nAb - nRt), base);
          st = ldz;
          k = (f == 0) ? 3 * (p - 1) : 3 * (f - 1) + 2;
        }
        if (full)
          s3_apply_seq<S3_K, true>(ptr, st, qmin, qmax, kb, tab + k, E);
        else
          s3_apply_seq<S3_K, false>(ptr, st, qmin, qmax, kb, tab + k, E);
      }
    }
    // (4) windows back to global memory.  Team mode: every CTA holds the same windows; the leader
    // writes them once all CTAs have finished reading the old ones (barrier), and the next batch
    // may only load after that (second barrier).
    if (cx.team) cx.sync();
    for (int e = tid; cx.lead && e < p * WW; e += nt) {
      const int f = e / WW, q = e - f * WW, r = q % S3_W, c = q / S3_W;
      if (r >= qmin && r <= qmax && c >= qmin && c <= qmax && (f == 0 || r <= c))
        stg_(&PSD_GE(cx.Hp(1 + f), ld, base + r, base + c), (f == 0 ? Xw : Dw + (size_t)(f - 1) * WW)[r + c * S3_W]);
    }
    cx.sync();
  }
}

// One double-shift sweep on the active block ifirst..ilast (order >= 3).
PSD_DEV void rq_double_shift_sweep(const GCtx<double>& cx, int ifirst, int ilast, int ifirstm, int ilastm,
                                   int iiter, int& nexc) {
  const int ld = cx.ldh;
  double* H1 = cx.Hp(1);
  double v0, v1, v2;
  if (iiter % 10 == 0) {
    nexc++;
    const double g = 0.6180339887498949;
    double fr[3];
    for (int m = 0; m < 3; m++) {
      const double x = (double)(3 * nexc + m + 1) * g;
      fr[m] = x - floor(x);
    }
    v0 = fr[0] + 0.25; v1 = fr[1] - 0.5; v2 = 0.5 * fr[2];
  } else {
    double Tl[3][3], Tt[3][3];
    int el, et;
    bool s1, s2;
    tri_block_product<3>(cx, ifirst, Tl, el, s1);
    tri_block_product<3>(cx, ilast - 2, Tt, et, s2);
    const int i = ifirst, k = ilast - 2, m = ilast - 1, nn = ilast;
    // leading entries of the product band (scale 2^el)
    const double a11 = PSD_GE(H1, ld, i, i), a12 = PSD_GE(H1, ld, i, i + 1);
    const double a21 = PSD_GE(H1, ld, i + 1, i), a22 = PSD_GE(H1, ld, i + 1, i + 1);
    const double a32 = PSD_GE(H1, ld, i + 2, i + 1);
    const double h11 = a11 * Tl[0][0], h21 = a21 * Tl[0][0];
    const double h12 = fma(a11, Tl[0][1], a12 * Tl[1][1]), h22 = fma(a21, Tl[0][1], a22 * Tl[1][1]);
    const double h32 = a32 * Tl[1][1];
    // trailing 2x2 of the product (scale 2^et), brought to the leading scale
    const double amk = PSD_GE(H1, ld, m, k), amm = PSD_GE(H1, ld, m, m), amn = PSD_GE(H1, ld, m, nn);
    const double anm = PSD_GE(H1, ld, nn, m), ann = PSD_GE(H1, ld, nn, nn);
    const double sc = scalbn(1.0, max(-600, min(600, et - el)));
    double h33 = fma(amk, Tt[0][1], amm * Tt[1][1]) * sc;
    double h34 = fma(amk, Tt[0][2], fma(amm, Tt[1][2], amn * Tt[2][2])) * sc;
    double h43 = anm * Tt[1][1] * sc;
    double h44 = fma(anm, Tt[1][2], ann * Tt[2][2]) * sc;
    // dlahqr-style shifts (PeriodicSchurDecompositions.jl:730-762) and first column (:768-803)
    double rt1r, rt2r, rt1i, rt2i;
    double s = fabs(h33) + fabs(h34) + fabs(h43) + fabs(h44);
    if (s == 0.0 || !isfinite(s)) {
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
    if (s == 0.0 || !isfinite(s)) {
      v0 = 1.0; v1 = 1.0; v2 = 1.0;
    } else {
      const double h21s = h21 / s;
      v0 = h21s * h12 + (h11 - rt1r) * ((h11 - rt2r) / s) - rt1i * (rt2i / s);
      v1 = h21s * (h11 + h22 - rt1r - rt2r);
      v2 = h21s * h32;
    }
  }
  {
    const double s = fabs(v0) + fabs(v1) + fabs(v2);
    if (s > 0.0 && isfinite(s)) { v0 /= s; v1 /= s; v2 /= s; } else { v0 = v1 = v2 = 1.0; }
  }
  Rot2 g;
  double r2, r1;
  givens_real(v1, v2, g.c2, g.s2, r2);
  givens_real(v0, r2, g.c1, g.s1, r1);
  if (cx.qzws >= 0 && ilast - ifirst - 1 >= 4) {
    if (cx.team)
      sweep_windowed<S3_K_TEAM>(cx, ifirst, ilast, ifirstm, ilastm, g, cx.qzws);
    else
      sweep_windowed<S3_K_CTA>(cx, ifirst, ilast, ifirstm, ilastm, g, cx.qzws);
  } else
  for (int j = ifirst; j <= ilast - 2; j++) {
    int zcol = 0;
    if (j > ifirst) {
      givens_real(PSD_GE(H1, ld, j + 1, j - 1), PSD_GE(H1, ld, j + 2, j - 1), g.c2, g.s2, r2);
      givens_real(PSD_GE(H1, ld, j, j - 1), r2, g.c1, g.s1, r1);
      zcol = j - 1;
    }
    chase_double(cx, j, g, zcol, r1, ilastm, ifirstm, min(j + 3, ilastm));
  }
  // trailing single rotation (:1015-1048)
  {
    const int j = ilast - 1;
    double c, s, r;
    givens_real(PSD_GE(H1, ld, j, j - 1), PSD_GE(H1, ld, j + 1, j - 1), c, s, r);
    chase_rotation<double>(cx, j, c, s, j - 1, r, j, ilastm, ifirstm, min(j + 2, ilastm));
  }
}

// ------------------------------------------------------------------------------------------
// Windowed single-shift sweep (complex path, factors in global memory): same organisation as
// sweep_windowed with one rotation per step.  Local index q <-> global index j0 - 1 + q; step s
// acts on q = s+1, s+2.  Rotations are tabulated in the bulk convention
// (a, b) <- (c a + s b, c b - conj(s) a).
// ------------------------------------------------------------------------------------------
template <class T>
struct S4 {
  // complex, C3 (128 registers per thread): K = 7 / 9 / 13 -> 1249 / 1263 / 1147 problems/s
  static constexpr int K = (sizeof(T) == sizeof(double)) ? 13 : 9;
  static constexpr int W = K + 3;
};
template <class T>
__host__ __device__ inline long long s4_work_scalars(int p) {
  return (long long)p * S4<T>::W * S4<T>::W + 2LL * S4<T>::K * (3 * (p - 1) + 3) + 8;
}

template <class T, bool FULL>
PSD_DEV void s4_apply_seq(T* ptr, long long stride, int qmin, int qmax, int kb, const double* rc, const T* rs, int E) {
  constexpr int K = S4<T>::K, W = S4<T>::W;
  T x[W];
  if (FULL) {
#pragma unroll
    for (int q = 0; q < W; q++) x[q] = ldg_(ptr + (long long)q * stride);
#pragma unroll
    for (int sx = 0; sx < K; sx++) {
      const double c = rc[sx * E];
      const T sv = rs[sx * E];
      const T a = x[sx + 1], b = x[sx + 2];
      x[sx + 1] = c * a + sv * b;
      x[sx + 2] = c * b - conj_(sv) * a;
    }
#pragma unroll
    for (int q = 0; q < W; q++) stg_(ptr + (long long)q * stride, x[q]);
    return;
  }
#pragma unroll
  for (int q = 0; q < W; q++)
    if (q >= qmin && q <= qmax) x[q] = ldg_(ptr + (long long)q * stride);
#pragma unroll
  for (int sx = 0; sx < K; sx++)
    if (sx < kb) {
      const double c = rc[sx * E];
      const T sv = rs[sx * E];
      const T a = x[sx + 1], b = x[sx + 2];
      x[sx + 1] = c * a + sv * b;
      x[sx + 2] = c * b - conj_(sv) * a;
    }
#pragma unroll
  for (int q = 0; q < W; q++)
    if (q >= qmin && q <= qmax) stg_(ptr + (long long)q * stride, x[q]);
}

// Steps j = ifirst .. ilast-1 of one single-shift sweep; (c, s) = the starting rotation.
template <class T>
PSD_DEV void sweep1_windowed(const GCtx<T>& cx, int ifirst, int ilast, int ifirstm, int ilastm, double c0, T s0,
                             long long ws_off) {
  constexpr int K = S4<T>::K, W = S4<T>::W, WW = W * W;
  const int n = cx.n, p = cx.p, tid = cx.tid, nt = cx.nt, ld = cx.ldh, ldz = cx.ldz;
  const int lane = tid & 31, warp = tid >> 5;
  const int E = 3 * (p - 1) + 3;
  T* Xw = reinterpret_cast<T*>(psd_smem_cq + ws_off);  // window of H_1, column-major, ld = W
  T* Dw = Xw + WW;                                      // windows of factors 2..p
  T* rs = Dw + (size_t)(p - 1) * WW;
  double* rc = reinterpret_cast<double*>(rs + (size_t)K * E);
  T* H1 = cx.Hp(1);
  const int nZ = cx.wantZ ? n : 0;
  for (int j0 = ifirst; j0 <= ilast - 1; j0 += K) {
    const int j1 = min(ilast - 1, j0 + K - 1), kb = j1 - j0 + 1;
    const int base = j0 - 1;
    const int qmin = (base >= ifirstm) ? 0 : 1;
    const int qmax = min(j1 + 2, ilast) - base;
    for (int e = tid; e < p * WW; e += nt) {
      const int f = e / WW, q = e - f * WW, r = q % W, c = q / W;
      if (r >= qmin && r <= qmax && c >= qmin && c <= qmax)
        (f == 0 ? Xw : Dw + (size_t)(f - 1) * WW)[r + c * W] = ldg_(&PSD_GE(cx.Hp(1 + f), ld, base + r, base + c));
    }
    __syncthreads();
    if (warp == 0) {
      for (int sx = 0; sx < kb; sx++) {
        const int j = j0 + sx, a = sx + 1;
        double c1 = c0;
        T s1 = s0;
        if (j > ifirst) {
          T r1;
          givens_chain(Xw[a + (a - 1) * W], Xw[a + 1 + (a - 1) * W], c1, s1, r1);
          __syncwarp();
          if (lane == 0) {
            Xw[a + (a - 1) * W] = r1;
            Xw[a + 1 + (a - 1) * W] = Scalar<T>::zero();
          }
        }
        if (lane >= a && lane <= qmax) {  // rows a, a+1 of the H_1 window
          T* pa = Xw + a + lane * W;
          const T x = pa[0], y = pa[1];
          pa[0] = c1 * x + s1 * y;
          pa[1] = c1 * y - conj_(s1) * x;
        }
        double ci = c1;
        T si = s1;
        for (int l = p; l >= 2; l--) {
          T* D = Dw + (size_t)(l - 2) * WW;
          RotChain<T> o;
          rot_chain_step<T>(cx.Sg(l), ci, si, D[a + a * W], D[a + (a + 1) * W], D[a + 1 + (a + 1) * W], o);
          __syncwarp();
          if (lane >= qmin && lane < a) {
            T* pa = D + lane + a * W;
            const T sv = conj_(o.sR), x = pa[0], y = pa[W];
            pa[0] = o.cR * x + sv * y;
            pa[W] = o.cR * y - conj_(sv) * x;
          } else if (lane >= a + 2 && lane <= qmax) {
            T* pa = D + a + lane * W;
            const T x = pa[0], y = pa[1];
            pa[0] = o.cL * x + o.sL * y;
            pa[1] = o.cL * y - conj_(o.sL) * x;
          } else if (lane == a) {
            D[a + a * W] = o.m00;
            D[a + (a + 1) * W] = o.m01;
            D[a + 1 + (a + 1) * W] = o.m11;
            const int k = sx * E + 3 * (l - 2);
            rc[k] = o.cR; rs[k] = conj_(o.sR);
            rc[k + 1] = o.cL; rs[k + 1] = o.sL;
            rc[k + 2] = o.co; rs[k + 2] = conj_(o.so);
          }
          __syncwarp();
          ci = o.co;
          si = o.so;
        }
        __syncwarp();
        if (lane >= qmin && lane <= min(a + 2, qmax)) {  // columns a, a+1 of the H_1 window
          T* pa = Xw + lane + a * W;
          const T sv = conj_(si), x = pa[0], y = pa[W];
          pa[0] = ci * x + sv * y;
          pa[W] = ci * y - conj_(sv) * x;
        }
        if (lane == 0) {
          const int k = sx * E + 3 * (p - 1);
          rc[k] = c1; rs[k] = s1;                // rows of H_1
          rc[k + 1] = c1; rs[k + 1] = conj_(s1);  // columns of Z_1
          rc[k + 2] = ci; rs[k + 2] = conj_(si);  // columns of H_1
        }
        __syncwarp();
      }
    }
    __syncthreads();
    {
      const int lo = base + qmin, hi = base + qmax;
      const int nAb = lo - ifirstm, nRt = ilastm - hi, per = nAb + nRt + nZ, total = p * per;
      const float rper = per > 0 ? 1.0f / (float)per : 0.0f;
      const bool full = (qmin == 0 && qmax == W - 1 && kb == K);
      for (int w = tid; w < total; w += nt) {
        int f, r;
        split_index(w, per, rper, f, r);  // f = 0: H_1 / Z_1, f >= 1: factor 1 + f
        T* ptr;
        long long st;
        int k;
        if (r < nAb) {
          ptr = &PSD_GE(cx.Hp(1 + f), ld, ifirstm + r, base);
          st = ld;
          k = (f == 0) ? 3 * (p - 1) + 2 : 3 * (f - 1);
        } else if (r < nAb + nRt) {
          ptr = &PSD_GE(cx.Hp(1 + f), ld, base, hi + 1 + (r - nAb));
          st = 1;
          k = (f == 0) ? 3 * (p - 1) : 3 * (f - 1) + 1;
        } else {
          ptr = &PSD_GE(cx.Zp(1 + f), ldz, 1 + (r - nAb - nRt), base);
          st = ldz;
          k = (f == 0) ? 3 * (p - 1) + 1 : 3 * (f - 1) + 2;
        }
        if (full)
          s4_apply_seq<T, true>(ptr, st, qmin, qmax, kb, rc + k, rs + k, E);
        else
          s4_apply_seq<T, false>(ptr, st, qmin, qmax, kb, rc + k, rs + k, E);
      }
    }
    for (int e = tid; e < p * WW; e += nt) {
      const int f = e / WW, q = e - f * WW, r = q % W, c = q / W;
      if (r >= qmin && r <= qmax && c >= qmin && c <= qmax && (f == 0 || r <= c))
        stg_(&PSD_GE(cx.Hp(1 + f), ld, base + r, base + c), (f == 0 ? Xw : Dw + (size_t)(f - 1) * WW)[r + c * W]);
    }
    __syncthreads();
  }
}

// Single-shift sweep of the complex periodic QZ iteration (generalized.jl:770-854).
PSD_DEV void cq_single_shift_sweep(const GCtx<cplx>& cx, int ifirst, int ilast, int ifirstm, int ilastm,
                                   int iiter, int& nexc) {
  const int p = cx.p, ld = cx.ldh;
  cplx* H1 = cx.Hp(1);

      double c;
      cplx s, r;
      if (iiter % 10 == 0) {
        nexc++;
        const double g = 0.6180339887498949;
        double fr[4];
        for (int m = 0; m < 4; m++) {
          const double x = (double)(4 * nexc + m + 1) * g;
          fr[m] = x - floor(x);
        }
        givens_t(mk(fr[0], fr[1]), mk(fr[2], fr[3]), c, s, r);
      } else {
        givens_t(mk(1.0, 0.0), mk(1.0, 0.0), c, s, r);
        for (int l = p; l >= 2; l--) {
          const cplx* Hl = cx.Hp(l);
          const cplx hf = PSD_GE(Hl, ld, ifirst, ifirst), hl = PSD_GE(Hl, ld, ilast, ilast);
          if (cx.Sg(l)) {
            givens_t(c * hf, hl * conj_(s), c, s, r);
          } else {
            givens_t(c * hl, -(hf * conj_(s)), c, s, r);
            s = -s;
          }
        }
        const cplx f = c * PSD_GE(H1, ld, ifirst, ifirst) - PSD_GE(H1, ld, ilast, ilast) * conj_(s);
        const cplx g = c * PSD_GE(H1, ld, ifirst + 1, ifirst);
        givens_t(f, g, c, s, r);
      }
      if (cx.qzws >= 0 && ilast - ifirst >= 4) {
        sweep1_windowed<cplx>(cx, ifirst, ilast, ifirstm, ilastm, c, s, cx.qzws);
        return;
      }
      for (int j = ifirst; j <= ilast - 1; j++) {
        int zcol = 0;
        if (j > ifirst) {
          givens_t(PSD_GE(H1, ld, j, j - 1), PSD_GE(H1, ld, j + 1, j - 1), c, s, r);
          zcol = j - 1;
        }
        chase_rotation(cx, j, c, s, zcol, r, j, ilastm, ifirstm, min(j + 2, ilastm));
      }
}

// generalized.jl:166-931.  Returns info (0 or the level ilast at which convergence failed).
template <class T>
PSD_DEV int gpqz_cta(const GCtx<T>& cx, const GqState<T>& st, bool wantT, int maxitfac, cplx* alpha,
                     T* beta, long long* scale) {
  constexpr bool kCplx = (sizeof(T) == sizeof(cplx));
  const int n = cx.n, p = cx.p, ld = cx.ldh, tid = cx.tid;
  const bool wantZ = cx.wantZ;
  T* H1 = cx.Hp(1);
  const double ulp = DBL_EPSILON;
  const double smlnum = DBL_MIN * ((double)n / ulp);
  const double safmin = DBL_MIN;
  const T czero = Scalar<T>::zero();
  // ziter = -1 when p >= log2(floatmin)/log2(eps) (~19.65)  (:199)
  int ziter = ((double)p >= (-1022.0) / (-52.0)) ? -1 : 0;
  int ilast = n, ifirst = -1, ifirstm = 1, ilastm = n, iiter = 1;
  int n2x2 = 0;  // consecutive attempts on the same 2x2 block (real path)
  const int maxit = maxitfac * n;
  int nexc = 0;
  bool done = false;

  for (int jiter = 1; jiter <= maxit; jiter++) {
    bool split1 = false, dpos = false, dneg = false, doqz = true;
    int ldef = -1, jdef = -1, jlo = 1;
    if (ilast == 1) {
      split1 = true;
    } else {
      split1 = cq_check_hess(cx, st, 1, ilast, ulp, smlnum, jlo);
      if (!split1) {
        dpos = cq_check_tr(cx, st, true, jlo, ilast, ulp, smlnum, ldef, jdef);
        if (!dpos) dneg = cq_check_tr(cx, st, false, jlo, ilast, ulp, smlnum, ldef, jdef);
        if (!dpos && !dneg && (ziter >= 7 || ziter < 0)) {
          // ---- Test 4: controlled zero shift (:356-448) ----
          for (int j = jlo; j <= ilast - 1; j++) {
            double c;
            T s;
            g_gen(cx, H1, ld, j, j, j + 1, j, c, s);
            g_lmul(cx, H1, ld, j, j + 1, c, s, j + 1, ilastm);
            CQ_SETG(j, c, s);
          }
          __syncthreads();
          if (wantZ) cq_rmul_seq(cx, st, cx.Zp(1), cx.ldz, jlo, ilast - 1, 1, 0, 1);
          for (int l = p; l >= 2; l--) {
            T* Hl = cx.Hp(l);
            for (int j = jlo; j <= ilast - 1; j++) {
              double c = st.Gc[j];
              T s = st.Gs[j];
              if (is_zero(s)) continue;
              if (cx.Sg(l))
                g_rmul(cx, Hl, ld, j, j + 1, c, s, ifirstm, j + 1);
              else
                g_lmul(cx, Hl, ld, j, j + 1, c, s, j, ilastm);
              double tol = abs_(PSD_GE(Hl, ld, j, j)) + abs_(PSD_GE(Hl, ld, j + 1, j + 1));
              if (tol == 0.0) tol = g_opnorm1(Hl, ld, jlo, j + 1, jlo, j + 1, false);
              tol = fmax(ulp * tol, smlnum);
              const bool small = abs_(PSD_GE(Hl, ld, j + 1, j)) <= tol;
              cx.sync();
              if (small) {
                if (cx.lead && tid == 0) PSD_GE(Hl, ld, j + 1, j) = czero;
                CQ_SETG(j, 1.0, czero);
                cx.sync();
              } else if (cx.Sg(l)) {
                g_gen(cx, Hl, ld, j, j, j + 1, j, c, s);
                g_lmul(cx, Hl, ld, j, j + 1, c, s, j + 1, ilastm);
                CQ_SETG(j, c, s);
              } else {
                g_gen(cx, Hl, ld, j + 1, j + 1, j + 1, j, c, s);
                g_rmul(cx, Hl, ld, j + 1, j, c, conj_(s), ifirstm, j);
                CQ_SETG(j, c, -s);
              }
            }
            __syncthreads();
            if (wantZ) cq_rmul_seq(cx, st, cx.Zp(l), cx.ldz, jlo, ilast - 1, 1, 0, 1);
          }
          ziter = 0;
          for (int j = jlo; j <= ilast - 1; j++) {
            const double c = st.Gc[j];
            const T s = st.Gs[j];
            g_rmul(cx, H1, ld, j, j + 1, c, s, ifirstm, j + 1);
            if (is_zero(s)) ziter = 1;
          }
          doqz = false;
        }
      }
    }

    if (dpos) {
      // ---- Case II: zero on the diagonal of an S+ factor: two unshifted half-sweeps (:453-566)
      for (int j = jlo; j <= jdef - 1; j++) {
        double c;
        T s;
        g_gen(cx, H1, ld, j, j, j + 1, j, c, s);
        g_lmul(cx, H1, ld, j, j + 1, c, s, j + 1, ilastm);
        CQ_SETG(j, c, s);
      }
      __syncthreads();
      if (wantZ) cq_rmul_seq(cx, st, cx.Zp(1), cx.ldz, jlo, jdef - 1, 1, 0, 1);
      for (int l = p; l >= 2; l--) {
        const int ntra = (l < ldef) ? (jdef - 2) : (jdef - 1);
        T* Hl = cx.Hp(l);
        for (int j = jlo; j <= ntra; j++) {
          double c = st.Gc[j];
          T s = st.Gs[j];
          if (cx.Sg(l)) {
            g_rmul(cx, Hl, ld, j, j + 1, c, s, ifirstm, j + 1);
            g_gen(cx, Hl, ld, j, j, j + 1, j, c, s);
            g_lmul(cx, Hl, ld, j, j + 1, c, s, j + 1, ilastm);
            CQ_SETG(j, c, s);
          } else {
            g_lmul(cx, Hl, ld, j, j + 1, c, s, j, ilastm);
            g_gen(cx, Hl, ld, j + 1, j + 1, j + 1, j, c, s);
            g_rmul(cx, Hl, ld, j + 1, j, c, conj_(s), ifirstm, j);
            CQ_SETG(j, c, -s);
          }
        }
        __syncthreads();
        if (wantZ) cq_rmul_seq(cx, st, cx.Zp(l), cx.ldz, jlo, ntra, 1, 0, 1);
      }
      for (int j = jlo; j <= jdef - 2; j++)
        g_rmul(cx, H1, ld, j, j + 1, st.Gc[j], st.Gs[j], ifirstm, j + 1);
      // second unshifted step, from the bottom (:512-564)
      for (int j = ilast; j >= jdef + 1; j--) {
        double c;
        T s;
        g_gen(cx, H1, ld, j, j, j, j - 1, c, s);
        g_rmul(cx, H1, ld, j, j - 1, c, conj_(s), ifirstm, j - 1);
        CQ_SETG(j, c, -s);
      }
      __syncthreads();
      if (wantZ) cq_rmul_seq(cx, st, cx.Zp(p > 1 ? 2 : 1), cx.ldz, ilast, jdef + 1, -1, -1, 0);
      for (int l = 2; l <= p; l++) {
        const int ntra = (l > ldef) ? (jdef + 2) : (jdef + 1);
        T* Hl = cx.Hp(l);
        for (int j = ilast; j >= ntra; j--) {
          double c = st.Gc[j];
          T s = st.Gs[j];
          if (!cx.Sg(l)) {
            g_rmul(cx, Hl, ld, j - 1, j, c, s, ifirstm, j);
            g_gen(cx, Hl, ld, j - 1, j - 1, j, j - 1, c, s);
            g_lmul(cx, Hl, ld, j - 1, j, c, s, j, ilastm);
            CQ_SETG(j, c, s);
          } else {
            g_lmul(cx, Hl, ld, j - 1, j, c, s, j - 1, ilastm);
            g_gen(cx, Hl, ld, j, j, j, j - 1, c, s);
            g_rmul(cx, Hl, ld, j, j - 1, c, conj_(s), ifirstm, j - 1);
            CQ_SETG(j, c, -s);
          }
        }
        __syncthreads();
        if (wantZ) cq_rmul_seq(cx, st, cx.Zp((l % p) + 1), cx.ldz, ilast, ntra, -1, -1, 0);
      }
      for (int j = ilast; j >= jdef + 2; j--)
        g_lmul(cx, H1, ld, j - 1, j, st.Gc[j], st.Gs[j], j - 1, ilastm);
      doqz = false;
    } else if (dneg) {
      // ---- Case III: zero on the diagonal of an S- factor (:568-740) ----
      T* Hd = cx.Hp(ldef);
      double c;
      T s;
      if (2 * jdef > (ilast - jlo + 1)) {  // bottom half: chase the zero down
        for (int j1 = jdef; j1 <= ilast - 1; j1++) {
          int j = j1;
          g_gen(cx, Hd, ld, j, j + 1, j + 1, j + 1, c, s);
          g_lmul(cx, Hd, ld, j, j + 1, c, s, j + 2, ilastm);
          int ln = (ldef % p) + 1;
          if (wantZ) g_rmul(cx, cx.Zp(ln), cx.ldz, j, j + 1, c, s, 1, n);
          int gi = j, gj = j + 1;
          for (int l = 1; l <= p - 1; l++) {
            if (ln == 1) {
              g_lmul(cx, H1, ld, gi, gj, c, s, j - 1, ilastm);
              g_gen(cx, H1, ld, j + 1, j, j + 1, j - 1, c, s);
              g_rmul(cx, H1, ld, j, j - 1, c, conj_(s), ifirstm, j);
              s = -s;
              gi = j - 1; gj = j;
              j -= 1;
            } else if (cx.Sg(ln)) {
              T* Hn = cx.Hp(ln);
              g_lmul(cx, Hn, ld, gi, gj, c, s, j, ilastm);
              g_gen(cx, Hn, ld, j + 1, j + 1, j + 1, j, c, s);
              g_rmul(cx, Hn, ld, j + 1, j, c, conj_(s), ifirstm, j);
              s = -s;
              gi = j; gj = j + 1;
            } else {
              T* Hn = cx.Hp(ln);
              g_rmul(cx, Hn, ld, gi, gj, c, s, ifirstm, j + 1);
              g_gen(cx, Hn, ld, j, j, j + 1, j, c, s);
              g_lmul(cx, Hn, ld, j, j + 1, c, s, j + 1, ilastm);
              gi = j; gj = j + 1;
            }
            ln = (ln % p) + 1;
            if (wantZ) g_rmul(cx, cx.Zp(ln), cx.ldz, gi, gj, c, s, 1, n);
          }
          g_rmul(cx, Hd, ld, gi, gj, c, s, ifirstm, j);
        }
        // deflate the last element in the Hessenberg factor (:620-655)
        const int j = ilast;
        g_gen(cx, H1, ld, j, j, j, j - 1, c, s);
        g_rmul(cx, H1, ld, j, j - 1, c, conj_(s), ifirstm, j - 1);
        s = -s;
        if (wantZ) g_rmul(cx, cx.Zp(p > 1 ? 2 : 1), cx.ldz, j - 1, j, c, s, 1, n);
        for (int l = 2; l <= ldef - 1; l++) {
          T* Hl = cx.Hp(l);
          if (!cx.Sg(l)) {
            g_rmul(cx, Hl, ld, j - 1, j, c, s, ifirstm, j);
            g_gen(cx, Hl, ld, j - 1, j - 1, j, j - 1, c, s);
            g_lmul(cx, Hl, ld, j - 1, j, c, s, j, ilastm);
          } else {
            g_lmul(cx, Hl, ld, j - 1, j, c, s, j - 1, ilastm);
            g_gen(cx, Hl, ld, j, j, j, j - 1, c, s);
            g_rmul(cx, Hl, ld, j, j - 1, c, conj_(s), ifirstm, j - 1);
            s = -s;
          }
          if (wantZ) g_rmul(cx, cx.Zp((l % p) + 1), cx.ldz, j - 1, j, c, s, 1, n);
        }
        g_rmul(cx, Hd, ld, j - 1, j, c, s, ifirstm, j);
      } else {  // top half: chase the zero up (:656-739)
        for (int j1 = jdef; j1 >= jlo + 1; j1--) {
          int j = j1;
          g_gen(cx, Hd, ld, j - 1, j, j - 1, j - 1, c, s);
          g_rmul(cx, Hd, ld, j, j - 1, c, conj_(s), ifirstm, j - 2);
          s = -s;
          if (wantZ) g_rmul(cx, cx.Zp(ldef), cx.ldz, j - 1, j, c, s, 1, n);
          int gi = j - 1, gj = j;
          int ln = ldef - 1;
          for (int l = 1; l <= p - 1; l++) {
            T* Hn = cx.Hp(ln);
            if (ln == 1) {
              g_rmul(cx, Hn, ld, gi, gj, c, s, ifirstm, j + 1);
              g_gen(cx, Hn, ld, j, j - 1, j + 1, j - 1, c, s);
              g_lmul(cx, Hn, ld, j, j + 1, c, s, j, ilastm);
              gi = j; gj = j + 1;
              j += 1;
            } else if (!cx.Sg(ln)) {
              g_lmul(cx, Hn, ld, gi, gj, c, s, j - 1, ilastm);
              g_gen(cx, Hn, ld, j, j, j, j - 1, c, s);
              g_rmul(cx, Hn, ld, j, j - 1, c, conj_(s), ifirstm, j - 1);
              s = -s;
              gi = j - 1; gj = j;
            } else {
              g_rmul(cx, Hn, ld, gi, gj, c, s, ifirstm, j);
              g_gen(cx, Hn, ld, j - 1, j - 1, j, j - 1, c, s);
              g_lmul(cx, Hn, ld, j - 1, j, c, s, j, ilastm);
              gi = j - 1; gj = j;
            }
            if (wantZ) g_rmul(cx, cx.Zp(ln), cx.ldz, gi, gj, c, s, 1, n);
            ln = (ln == 1) ? p : (ln - 1);
          }
          g_lmul(cx, Hd, ld, gi, gj, c, s, j, ilastm);
        }
        // deflate the first element in the Hessenberg factor (:705-738)
        const int j = jlo;
        g_gen(cx, H1, ld, j, j, j + 1, j, c, s);
        g_lmul(cx, H1, ld, j, j + 1, c, s, j + 1, ilastm);
        if (wantZ) g_rmul(cx, cx.Zp(1), cx.ldz, j, j + 1, c, s, 1, n);
        for (int l = p; l >= ldef + 1; l--) {
          T* Hl = cx.Hp(l);
          if (cx.Sg(l)) {
            g_rmul(cx, Hl, ld, j, j + 1, c, s, ifirstm, j + 1);
            g_gen(cx, Hl, ld, j, j, j + 1, j, c, s);
            g_lmul(cx, Hl, ld, j, j + 1, c, s, j + 1, ilastm);
          } else {
            g_lmul(cx, Hl, ld, j, j + 1, c, s, j, ilastm);
            g_gen(cx, Hl, ld, j + 1, j + 1, j + 1, j, c, s);
            g_rmul(cx, Hl, ld, j + 1, j, c, conj_(s), ifirstm, j);
            s = -s;
          }
          if (wantZ) g_rmul(cx, cx.Zp(l), cx.ldz, j, j + 1, c, s, 1, n);
        }
        g_lmul(cx, Hd, ld, j, j + 1, c, s, j + 1, ilastm);
      }
      doqz = false;
    } else if (split1) {
      // ---- 1x1 block split off (:741-762) ----
      if (cx.lead && tid == 0) {
        T a;
        int b;
        long long sc;
        safeprod<T>(p, cx.S, [&](int l) { return PSD_GE(cx.Hp(l), ld, ilast, ilast); }, a, b, sc);
        alpha[ilast - 1] = mk(re_(a), im_(a));
        beta[ilast - 1] = Scalar<T>::from_real((double)b);
        scale[ilast - 1] = sc;
      }
      ilast -= 1;
      if (ilast < 1) {
        done = true;
        break;
      }
      iiter = 0;
      if (ziter != -1) ziter = 0;
      if (!wantT) {
        ilastm = ilast;
        if (ifirstm > ilast) ifirstm = 1;
      }
      doqz = false;
    } else if (doqz) {
      ifirst = jlo;
    }

    if (doqz) {
      iiter++;
      ziter++;
      if (!wantT) ifirstm = ifirst;
      if constexpr (kCplx) {
        cq_single_shift_sweep(cx, ifirst, ilast, ifirstm, ilastm, iiter, nexc);
      } else {
        // ---- real path: 2x2 block handling / double-shift sweep (rgeneralized.jl:655-1054) ----
        if (ifirst + 1 == ilast) {
          n2x2++;
          if (rq_block2x2(cx, ifirst, ifirstm, ilastm, n2x2 > 20, alpha, beta, scale)) {
            // complex pair (or accepted block) split off (:748-790)
            n2x2 = 0;
            ilast = ifirst - 1;
            if (ilast < 1) {
              done = true;
              break;
            }
            iiter = 0;
            if (ziter != -1) ziter = 0;
            if (!wantT) {
              ilastm = ilast;
              if (ifirstm > ilast) ifirstm = 1;
            }
          }
        } else {
          n2x2 = 0;
          rq_double_shift_sweep(cx, ifirst, ilast, ifirstm, ilastm, iiter, nexc);
        }
      }
    }
  }
  if (!done) return ilast;  // "convergence failed at level ilast" (:856-858)

  if constexpr (kCplx) {
   if (wantT) {
    // ---- make diag(H_l), l >= 2, real non-negative (:860-908) ----
    for (int l = p; l >= 2; l--) {
      cplx* Hl = cx.Hp(l);
      cplx* Hm = cx.Hp(l - 1);
      cplx* Zl = wantZ ? cx.Zp(l) : nullptr;
      const bool sl = cx.Sg(l), sm = cx.Sg(l - 1);
      // scalefacs[j] -> Gs[j] (reuse), computed by one thread per j
      for (int j = 1 + tid; j <= n; j += cx.nt) {
        const cplx d = PSD_GE(Hl, ld, j, j);
        const double abst = abs_(d);
        cplx z = mk(1.0, 0.0);
        if (abst > safmin) z = conj_(d / abst);
        st.Gs[j] = sl ? z : conj_(z);
        st.Gc[j] = (abst > safmin) ? abst : -1.0;
      }
      __syncthreads();
      for (int e = cx.wtid; e < n * n; e += cx.wnt) {
        const int r0 = 1 + e % n, c0 = 1 + e / n;
        // this factor
        if (sl) {
          // row j scaled by z_j right of the diagonal
          if (c0 > r0 && st.Gc[r0] >= 0.0) PSD_GE(Hl, ld, r0, c0) = PSD_GE(Hl, ld, r0, c0) * st.Gs[r0];
        } else {
          // column j scaled by z_j = conj(scalefacs[j]) above the diagonal
          if (r0 < c0 && st.Gc[c0] >= 0.0) PSD_GE(Hl, ld, r0, c0) = PSD_GE(Hl, ld, r0, c0) * conj_(st.Gs[c0]);
        }
        if (r0 == c0 && st.Gc[r0] >= 0.0) PSD_GE(Hl, ld, r0, c0) = mk(st.Gc[r0], 0.0);
        if (Zl) PSD_GE(Zl, cx.ldz, r0, c0) = PSD_GE(Zl, cx.ldz, r0, c0) * conj_(st.Gs[c0]);
        if (sm) {
          if (r0 <= c0) PSD_GE(Hm, ld, r0, c0) = PSD_GE(Hm, ld, r0, c0) * conj_(st.Gs[c0]);
        } else {
          if (c0 >= r0) PSD_GE(Hm, ld, r0, c0) = PSD_GE(Hm, ld, r0, c0) * st.Gs[r0];
        }
      }
      cx.sync();
    }
  }
  }
  return 0;
}


// Factors whose largest entry lies outside [2^-500, 2^500] are scaled by an exact power of two into
// [0.5, 1) before the reduction: the QZ's absolute thresholds (safmin / ulp) take an inverted factor
// near 1e-300 for a singular one, and subnormal or near-overflow factors do not converge.  ex[l-1]
// receives the exponent e_l (factor l was multiplied by 2^-e_l; 0: left as it was) and the return
// value is the shift of the eigenvalues, sum over l of s_l ? e_l : -e_l.  Factors inside the window
// are not touched, so results on them are the same bit for bit.  All threads of the CTA call this;
// `cell` is one word of shared memory for the reduction.
template <class T>
__device__ __noinline__ long long factor_scale_exponents(const GCtx<T>& cx, int* ex, long long* cell) {
  const int n = cx.n, p = cx.p, tid = cx.tid, nt = cx.nt;
  long long shift = 0;
  for (int l = 1; l <= p; l++) {
    T* Hl = cx.Hp(l);
    double m = 0.0;
    for (int e = tid; e < n * n; e += nt) m = fmax(m, fmax(fabs(re_(Hl[(e % n) + (size_t)(e / n) * cx.ldh])),
                                                           fabs(im_(Hl[(e % n) + (size_t)(e / n) * cx.ldh]))));
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (tid == 0) *cell = 0;
    __syncthreads();
    // the bit patterns of non-negative doubles order as the values do
    if ((tid & 31) == 0) atomicMax(cell, __double_as_longlong(m));
    __syncthreads();
    m = __longlong_as_double(*cell);
    __syncthreads();
    int k = 0;
    if (m > 0.0 && isfinite(m) && (m < 0x1p-500 || m > 0x1p500)) (void)frexp(m, &k);
    if (k != 0)
      for (int e = tid; e < n * n; e += nt) {
        T& x = Hl[(e % n) + (size_t)(e / n) * cx.ldh];
        x = scal2(x, -k);
      }
    if (tid == 0) ex[l - 1] = k;
    shift += cx.Sg(l) ? k : -k;
  }
  __syncthreads();
  return shift;
}

// Undoes factor_scale_exponents: the eigenvalues (finite, non-zero; al == nullptr: none) by
// 2^eshift, factor l of T by 2^e_l.
template <class T>
__device__ __noinline__ void undo_factor_scale(const GCtx<T>& cx, const int* ex, long long eshift, const cplx* al,
                                               const T* be, long long* sc) {
  const int n = cx.n, tid = cx.tid, nt = cx.nt;
  if (al && eshift != 0)
    for (int i = tid; i < n; i += nt)
      if (!is_zero(be[i]) && !(al[i].x == 0.0 && al[i].y == 0.0)) sc[i] += eshift;
  for (int l = 1; l <= cx.p; l++) {
    const int k = ex[l - 1];
    if (k == 0) continue;
    T* Hl = cx.Hp(l);
    for (int e = tid; e < n * n; e += nt) {
      T& x = Hl[(e % n) + (size_t)(e / n) * cx.ldh];
      x = scal2(x, k);
    }
  }
}

template <class T, int MAXT>
__global__ void __launch_bounds__(MAXT, 1) gpschur_kernel(GpqzParams<T> P) {
  const int n = P.n, p = P.p, tid = threadIdx.x, nt = blockDim.x;
  const size_t nn = (size_t)n * n;
  __shared__ long long s_b;
  __shared__ int s_key;

  double* small = psd_smem_cq;
  GqState<T> st;
  st.Gc = small;
  st.Gs = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1));
  T* stage = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1) + 2 * (n + 2));
  T* stage_in = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1) + 2 * (n + 2) + cq_stage_doubles(p));
  T* wvec = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1) + 2 * (n + 2) + 2 * cq_stage_doubles(p));
  unsigned char* Sint = reinterpret_cast<unsigned char*>(small + (n + 2) + ((n + 2) & 1) + 4 * (n + 2) +
                                                         2 * cq_stage_doubles(p));
  st.key = &s_key;
  T* mats = reinterpret_cast<T*>(psd_smem_cq + ((cq_small_doubles(n, p) + 1) & ~1LL));

  const bool left = P.left != 0;
  // internal signature: reversed for :L (generalized.jl:114-123)
  for (int l = tid; l < p; l += nt) Sint[l] = P.S[left ? (p - 1 - l) : l];
  __syncthreads();

  GCtx<T> cx;
  cx.n = n; cx.p = p; cx.tid = tid; cx.nt = nt;
  cx.wantZ = P.wantZ && P.Z;
  cx.S = Sint;
  cx.stage = stage;
  cx.stage_in = stage_in;
  cx.wvec = wvec;
  cx.wtid = tid; cx.wnt = nt; cx.lead = true; cx.team = false;
  cx.blk = P.blocked_stage1 ? mats : nullptr;  // global mode: the matrix area of smem is free
  cx.rots = P.deep ? small + cq_rots_offset(n, p) : nullptr;
  cx.deep_u = P.deep;
  cx.s2ws = P.windowed_stage2 ? ((cq_small_doubles(n, p) + 1) & ~1LL) : -1;
  cx.qzws = P.windowed_qz ? ((cq_small_doubles(n, p) + 1) & ~1LL) : -1;
  __shared__ long long s_prof[4];
  cx.prof = P.debug ? s_prof : nullptr;

  for (;;) {
    if (tid == 0) s_b = (long long)atomicAdd(P.counter, 1ULL);
    __syncthreads();
    const long long b = s_b;
    __syncthreads();
    if (b >= P.batch) break;
    T* Ab = P.A + (size_t)b * p * nn;
    T* Zb = cx.wantZ ? (P.Z + (size_t)b * p * nn) : nullptr;
    if (P.use_smem) {
      cx.ldh = P.ldh; cx.ldz = P.ldh;
      cx.H = mats; cx.hs = (long long)P.ldh * n;
      cx.Z = mats + (size_t)p * P.ldh * n; cx.zs = (long long)P.ldh * n;
      cx.zmap_left = false;
      for (int l = 1; l <= p; l++) {
        const T* src = Ab + (size_t)((left ? (p + 1 - l) : l) - 1) * nn;
        T* dst = cx.Hp(l);
        for (int e = tid; e < (int)nn; e += nt) dst[(e % n) + (size_t)(e / n) * cx.ldh] = src[e];
      }
    } else {
      cx.ldh = n; cx.ldz = n;
      if (left) {
        cx.H = Ab + (size_t)(p - 1) * nn; cx.hs = -(long long)nn;
      } else {
        cx.H = Ab; cx.hs = (long long)nn;
      }
      cx.Z = Zb; cx.zs = (long long)nn;
      cx.zmap_left = left;
    }
    __syncthreads();

    int* ex = P.pexp + (size_t)blockIdx.x * p;
    const long long eshift = factor_scale_exponents(cx, ex, &s_b);  // (s_b is free until the next problem)
    const long long tstart = clock64();
    if (!P.skip_reduce) {
      gphessenberg_cta(cx);
    } else {
      if (cx.wantZ) {
        for (int l = 1; l <= p; l++) {
          T* Zl = cx.Zp(l);
          for (int e = tid; e < (int)nn; e += nt)
            Zl[(e % n) + (size_t)(e / n) * cx.ldz] = ((e % n) == (e / n)) ? Scalar<T>::one() : Scalar<T>::zero();
        }
      }
    }
    // enforce exact Hessenberg / triangular structure (_gethess!, :195; triu! :1027)
    for (int l = 1; l <= p; l++) {
      T* Hl = cx.Hp(l);
      const int keep = (l == 1) ? 1 : 0;
      for (int e = tid; e < (int)nn; e += nt) {
        const int r = e % n, c = e / n;
        if (r > c + keep) Hl[r + (size_t)c * cx.ldh] = Scalar<T>::zero();
      }
    }
    __syncthreads();

    cplx* al = P.alpha + (size_t)b * n;
    T* be = P.beta + (size_t)b * n;
    long long* sc = P.scale + (size_t)b * n;
    const long long tred = clock64();
    const int info = P.reduce_only ? 0 : gpqz_cta<T>(cx, st, P.wantT != 0, P.maxitfac, al, be, sc);
    if (P.debug && tid == 0 && blockIdx.x == 0)
      printf("[psd gpschur b=%lld] stage1 %lld  stage2 %lld  qz %lld cycles\n", b,
             P.skip_reduce ? 0LL : s_prof[0] - tstart, P.skip_reduce ? 0LL : tred - s_prof[0], clock64() - tred);
    if (tid == 0) P.info[b] = info;
    __syncthreads();
    undo_factor_scale(cx, ex, eshift, P.reduce_only ? nullptr : al, be, sc);
    __syncthreads();

    if (P.use_smem) {
      if (P.wantT) {
        for (int l = 1; l <= p; l++) {
          T* dst = Ab + (size_t)((left ? (p + 1 - l) : l) - 1) * nn;
          const T* src = cx.Hp(l);
          for (int e = tid; e < (int)nn; e += nt) dst[e] = src[(e % n) + (size_t)(e / n) * cx.ldh];
        }
      }
      if (cx.wantZ) {
        for (int l = 1; l <= p; l++) {
          const int s = (left && l > 1) ? (p + 2 - l) : l;
          T* dst = Zb + (size_t)(s - 1) * nn;
          const T* src = cx.Zp(l);
          for (int e = tid; e < (int)nn; e += nt) dst[e] = src[(e % n) + (size_t)(e / n) * cx.ldz];
        }
      }
    }
    __syncthreads();
  }
}


// ---------------------------------------------------------------------------------------------
// Team kernel: ONE large problem at a time on the whole GPU (cooperative launch, one CTA per SM).
// Input must already be in Hessenberg-triangular form (the blocked reduction of
// psd_large_hess.cuh, or the inner pschur!(H1, Hs, S) entry); Z is either preset (the Q_j of the
// reduction) or initialised to the identity here.  Every CTA executes gpqz_cta redundantly; see
// GCtx for how the work is shared.  Factors and Z stay in place in global memory.
// ---------------------------------------------------------------------------------------------
template <class T>
__global__ void gpschur_team_kernel(GpqzParams<T> P, int z_preset) {
  namespace cgx = cooperative_groups;
  cgx::grid_group grid = cgx::this_grid();
  const int n = P.n, p = P.p, tid = threadIdx.x, nt = blockDim.x;
  const size_t nn = (size_t)n * n;
  __shared__ int s_key;
  double* small = psd_smem_cq;
  GqState<T> st;
  st.Gc = small;
  st.Gs = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1));
  T* stage = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1) + 2 * (n + 2));
  T* stage_in = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1) + 2 * (n + 2) + cq_stage_doubles(p));
  T* wvec = reinterpret_cast<T*>(small + (n + 2) + ((n + 2) & 1) + 2 * (n + 2) + 2 * cq_stage_doubles(p));
  unsigned char* Sint = reinterpret_cast<unsigned char*>(small + (n + 2) + ((n + 2) & 1) + 4 * (n + 2) +
                                                         2 * cq_stage_doubles(p));
  st.key = &s_key;
  const bool left = P.left != 0;
  for (int l = tid; l < p; l += nt) Sint[l] = P.S ? P.S[left ? (p - 1 - l) : l] : 1;
  __syncthreads();
  GCtx<T> cx;
  cx.n = n; cx.p = p; cx.tid = tid; cx.nt = nt;
  cx.wantZ = P.wantZ && P.Z;
  cx.S = Sint;
  cx.stage = stage; cx.stage_in = stage_in; cx.wvec = wvec; cx.prof = nullptr;
  cx.wtid = blockIdx.x * nt + tid; cx.wnt = gridDim.x * nt;
  cx.lead = blockIdx.x == 0; cx.team = true;
  cx.blk = nullptr;
  cx.rots = P.deep ? small + cq_rots_offset(n, p) : nullptr;
  cx.deep_u = P.deep;
  cx.s2ws = -1;
  cx.qzws = P.windowed_qz ? ((cq_small_doubles(n, p) + 1) & ~1LL) : -1;
  cx.ldh = n; cx.ldz = n;
  for (long long b = 0; b < P.batch; b++) {
    T* Ab = P.A + (size_t)b * p * nn;
    T* Zb = cx.wantZ ? (P.Z + (size_t)b * p * nn) : nullptr;
    if (left) {
      cx.H = Ab + (size_t)(p - 1) * nn; cx.hs = -(long long)nn;
    } else {
      cx.H = Ab; cx.hs = (long long)nn;
    }
    cx.Z = Zb; cx.zs = (long long)nn;
    cx.zmap_left = left;
    if (cx.wantZ && !z_preset)
      for (int l = 1; l <= p; l++) {
        T* Zl = cx.Zp(l);
        for (long long e = cx.wtid; e < (long long)nn; e += cx.wnt)
          Zl[e] = ((e % n) == (e / n)) ? Scalar<T>::one() : Scalar<T>::zero();
      }
    for (int l = 1; l <= p; l++) {
      T* Hl = cx.Hp(l);
      const int keep = (l == 1) ? 1 : 0;
      for (long long e = cx.wtid; e < (long long)nn; e += cx.wnt) {
        const int r = (int)(e % n), c = (int)(e / n);
        if (r > c + keep) Hl[e] = Scalar<T>::zero();
      }
    }
    grid.sync();
    const int info = gpqz_cta<T>(cx, st, P.wantT != 0, P.maxitfac, P.alpha + (size_t)b * n,
                                 P.beta + (size_t)b * n, P.scale + (size_t)b * n);
    if (cx.lead && tid == 0) P.info[b] = info;
    grid.sync();
  }
}

// (alpha, beta, alphascale) -> eigenvalue alpha / beta * 2^alphascale (generalized.jl:75-76); used
// when the real standard path runs its iteration on the generalized team kernel with S = trues.
__global__ void gvalues_kernel(const cplx* alpha, const double* beta, const long long* scale, double* eig,
                               long long count) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < count;
       e += (long long)gridDim.x * blockDim.x) {
    const long long sc = scale[e];
    const int s1 = (int)(sc / 2), s2 = (int)(sc - sc / 2);
    const double re = scalbn(scalbn(alpha[e].x / beta[e], s1), s2);
    const double im = scalbn(scalbn(alpha[e].y / beta[e], s1), s2);
    eig[2 * e] = re;
    eig[2 * e + 1] = (alpha[e].y == 0.0) ? 0.0 : im;
  }
}

}  // namespace psd
