// CUDA kernels of the large-N multishift periodic QR iteration (see psd_ms_core.cuh for the
// algorithm and psd_ms.cu for the host driver):
//   ms_chase_kernel      one CTA per diagonal window: stage the p windows in shared memory, chase
//                        the packet of bulges, accumulate U_j, write windows and U_j back
//   ms_apply_kernel      in-place tile updates  X <- U' X  /  X <- X U  on the FP64 tensor cores
//                        (DMMA m8n8k4) for the off-window parts of H_j and for Z_j
//   ms_scan_kernel       deflation scan of the subdiagonal of H_1, active block
//   ms_shifts_kernel     eigenvalues of the trailing window (periodic_qr_cta, eigenvalues only)
//   ms_blocklist_kernel / ms_blocks_kernel   final stage: every remaining diagonal block of order
//                        <= W is brought to (standardised) periodic Schur form by one CTA each
//   ms_maxabs / ms_scale  exact power-of-two normalisation of the factors (overflow safety)
#pragma once
#include <cuda_runtime.h>

#include "psd_ms_core.cuh"
#include "psd_real_qr.cuh"

namespace psd {
namespace ms {

extern __shared__ __align__(16) double ms_smem[];

// FP64 tensor-core instruction (SASS DMMA): D(8x8) += A(8x4) * B(4x8); per lane a = A[lane/4][lane%4],
// b = B[lane%4][lane/4], d0/d1 = D[lane/4][2*(lane%4) + 0/1].
__device__ __forceinline__ void ms_dmma(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

// ------------------------------------------------------------------------------------------
// Workspace layout (device): U_j of the window / block that starts at row s lives at
//   U + (j-1) * n * W + s * W,  column-major with leading dimension = order of the window.
// Windows that exist at the same time are disjoint in index space, so these never overlap.
// ------------------------------------------------------------------------------------------
constexpr int MS_SHIFT_SLOTS = 8;
constexpr int MS_SS_NP = 0, MS_SS_SEQ = MS_SHIFT_SLOTS, MS_SS_LO = 2 * MS_SHIFT_SLOTS;  // offsets into shift_state
constexpr int MS_SS_INTS = 3 * MS_SHIFT_SLOTS;
struct ChaseParams {
  int n, p;
  Geom g;
  double* H[MS_MAXP];  // internal factor j at H[j-1], column-major, ld = n
  double* U;
  const double* shifts;  // [slots][66][4] pair buffers
  const int* shift_state;  // per shift slot: number of pairs, sequence number (0: being computed), first source row
  const WinDesc* wins;   // this round's windows in mapped pinned host memory (written by the host)
  WinDesc* wins_dev;     // device copy made here for the update and scan kernels of the round
  int* idle_count;       // number of windows found idle (statistics), or nullptr
  long long* prof;       // [8] cycle counters of CTA 0 (debug), or nullptr
};

struct DevExec {
  static constexpr int LANES = 32;
  BState st;
  int b, role, lane;
  bool prof = false;
  long long tl = 0, acc[4] = {0, 0, 0, 0};
  template <class F>
  __device__ __forceinline__ void each(F&& f) { f(b, role, lane, st); }
  __device__ __forceinline__ void barrier() { __syncthreads(); }
  __device__ __forceinline__ void tick(int slot) {
    if (prof) {
      const long long t = clock64();
      acc[slot] += t - tl;
      tl = t;
    }
  }
};

__global__ void __launch_bounds__(64 * MS_MAXNB, 1) ms_chase_kernel(ChaseParams P) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const long long P_t0 = clock64();
  if (P.prof && blockIdx.x == 0 && tid == 0) {
    // debug: device-side gap between the end of the previous scan kernel and this kernel's start
    unsigned long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    const unsigned long long last = ((volatile unsigned long long*)P.prof)[15];
    if (last != 0 && now > last) atomicAdd((unsigned long long*)&P.prof[7], now - last);
  }
  __shared__ WinDesc s_desc;
  if (tid == 0) {
    s_desc = P.wins[blockIdx.x];
    if (s_desc.intro) {
      // newest complete shift set computed from rows of this window's block (free-running supply
      // on the side streams); failing that the newest complete set of any block; failing that
      // none (npairs = 0: unshifted start vector)
      const volatile int* ss = (const volatile int*)P.shift_state;
      int best = -1, bseq = 0, any = -1, aseq = 0;
      for (int k = 0; k < MS_SHIFT_SLOTS; k++) {
        const int sq = ss[MS_SS_SEQ + k];
        if (sq <= 0) continue;
        const int lo = ss[MS_SS_LO + k];
        if (lo >= s_desc.ilo && lo <= s_desc.ihi && sq > bseq) { best = k; bseq = sq; }
        if (sq > aseq) { any = k; aseq = sq; }
      }
      const int slot = best >= 0 ? best : any;
      s_desc.pair_off = slot >= 0 ? slot * 66 : 0;
      s_desc.npairs = slot >= 0 ? ss[MS_SS_NP + slot] : 0;
    }
    // T = 0: a packet held back by the drain (psd_ms_driver.hpp); only the scan reads the entry
    if (s_desc.T == 0) s_desc.idle = 1;
    P.wins_dev[blockIdx.x] = s_desc;
  }
  __syncthreads();
  const WinDesc d = s_desc;
  if (d.T == 0) return;
  const int W = P.g.W, LD = P.g.LD, p = P.p, n = P.n;
  Ctx c;
  c.p = p; c.W = W; c.LD = LD;
  c.Hw = ms_smem;
  c.Uw = ms_smem + (size_t)p * W * LD;
  c.mbox = ms_smem + (size_t)2 * p * W * LD;
  c.shifts = P.shifts;
  c.d = d;
  const int wl = d.wl, s = d.s;
  for (int j = 1; j <= p; j++) {
    const double* src = P.H[j - 1] + s + (size_t)s * n;
    double* dst = c.H(j);
    double* u = c.U(j);
    for (int e = tid; e < wl * wl; e += nt) {
      const int r = e % wl, cc = e / wl;
      dst[r + (size_t)cc * LD] = src[r + (size_t)cc * n];
      u[r + (size_t)cc * LD] = (r == cc) ? 1.0 : 0.0;
    }
  }
  __syncthreads();
  // deflations made since this window was planned (exact zeros on the subdiagonal of H_1)
  __shared__ int s_bihi[MS_MAXNB];
  c.bihi = s_bihi;
  if (tid < d.nbul) s_bihi[tid] = clamp_block_end(c, tid);
  __syncthreads();
  DevExec ex;
  ex.b = tid >> 6;
  ex.role = (tid >> 5) & 1;
  ex.lane = tid & 31;
  ex.st.active = 0;
  ex.prof = (P.prof != nullptr) && blockIdx.x == 0 && tid == 0;
  const long long tk0 = ex.prof ? clock64() : 0;
  ex.tl = tk0;
  chase_window(c, ex);
  __syncthreads();
  const long long tk1 = ex.prof ? clock64() : 0;
  int moved = 0;  // some U_j differs from the identity
  for (int j = 1; j <= p; j++) {
    double* dst = P.H[j - 1] + s + (size_t)s * n;
    const double* src = c.H(j);
    const double* u = c.U(j);
    double* ud = P.U + (size_t)(j - 1) * n * W + (size_t)s * W;
    for (int e = tid; e < wl * wl; e += nt) {
      const int r = e % wl, cc = e / wl;
      dst[r + (size_t)cc * n] = src[r + (size_t)cc * LD];
      const double uv = u[r + (size_t)cc * LD];
      ud[r + (size_t)cc * W] = uv;
      moved |= (uv != ((r == cc) ? 1.0 : 0.0));
    }
  }
  // a packet whose bulges have all been chased off leaves identities: tell the update kernels
  moved = __syncthreads_or(moved);
  if (tid == 0 && !moved) {
    P.wins_dev[blockIdx.x].idle = 1;
    if (P.idle_count) atomicAdd(P.idle_count, 1);
  }
  if (ex.prof) {
    __syncthreads();
    const long long tk2 = clock64();
    atomicAdd((unsigned long long*)&P.prof[0], (unsigned long long)ex.acc[1]);  // chain phases
    atomicAdd((unsigned long long*)&P.prof[1], (unsigned long long)ex.acc[2]);  // column phases
    atomicAdd((unsigned long long*)&P.prof[2], (unsigned long long)ex.acc[3]);  // row phases
    atomicAdd((unsigned long long*)&P.prof[3], (unsigned long long)(tk2 - tk1));  // write-back
    atomicAdd((unsigned long long*)&P.prof[4], (unsigned long long)(tk2 - P_t0));  // whole CTA
    atomicAdd((unsigned long long*)&P.prof[5], (unsigned long long)d.T);
    atomicAdd((unsigned long long*)&P.prof[6], 1ULL);
  }
}

// ------------------------------------------------------------------------------------------
// Deflation scan + active blocks.  ctl (device ints): [0] ilo, [1] ihi of the lowest active block,
// [2] done, [3] number of subdiagonal entries set to zero by this scan, [4] sequence number
// (written last), [5] number of active blocks reported (<= MS_MAXBLK, lowest first), [6 + 2 b],
// [7 + 2 b] first and last row of block b.
// Criterion: |h(k,k-1)| <= max(smlnum, ulp (|h(k-1,k-1)| + |h(k,k)|)) on H_1 (the "Test 1" of the
// periodic QZ drivers, rgeneralized.jl:1086-1112), which perturbs H_1 by at most 2 ulp ||H_1||.
// Active blocks: the unreduced diagonal blocks of order > nmin.
// ------------------------------------------------------------------------------------------
// The rows of the bulge chains that sit in the matrix after the round (wins[0..nwin), see
// chain_after_round) are left alone: subdiagonal entries there are part of the bulges.
// Dynamic shared memory: 2 n bytes (skip flags, non-zero flags of the subdiagonal).
constexpr int MS_MAXCHAINS = 160;
constexpr int MS_SCAN_CAND = 256;  // candidate blocks kept by the scan before the lowest MS_MAXBLK are reported
constexpr int MS_SCAN_INTS = 6 + 2 * MS_MAXBLK + 2;  // ints per scan result (see ms_scan_body)

// The result (ctl[0..3]) and then the sequence number ctl[4] stay in device memory; the host polls
// for them with copies on a side stream.
__device__ __forceinline__ void ms_scan_body(double* H1, int n, int nmin, int* ctl, int seq, const WinDesc* wins,
                                             int nwin, int W, int D, long long* prof, unsigned char* smem_bytes) {
  __shared__ int s_cnt;
  unsigned char* skip = smem_bytes;  // skip[z]: entry H1[z+1, z] belongs to a chain
  unsigned char* nz = skip + n;                                      // nz[k]: H1[k, k-1] != 0 (k >= 1)
  const int tid = threadIdx.x, nt = blockDim.x;
  if (tid == 0) s_cnt = 0;
  for (int k = tid; k < n; k += nt) skip[k] = 0;
  __syncthreads();
  if (nwin > MS_MAXCHAINS) nwin = MS_MAXCHAINS;  // (the host never plans more)
  for (int e = tid; e < nwin * 32; e += nt) {
    const int w = e >> 5, o = e & 31;
    int a = 1, b = 0;
    if (chain_after_round(wins[w], W, D, a, b)) {
      const int z = a + o;  // a chain covers at most 3 NB + 3 <= 27 entries
      if (z <= b && z >= 0 && z < n) skip[z] = 1;
    }
  }
  __syncthreads();
  const double smlnum = DBL_MIN * ((double)n / DBL_EPSILON);
  int cnt = 0;
  for (int k = 1 + tid; k < n; k += nt) {
    double* e = H1 + k + (size_t)(k - 1) * n;
    double sub = *e;
    if (sub != 0.0 && !skip[k - 1] &&
        ms_negligible(sub, H1[(k - 1) + (size_t)(k - 1) * n], H1[k + (size_t)k * n], smlnum)) {
      *e = 0.0;
      sub = 0.0;
      cnt++;
    }
    nz[k] = (sub != 0.0);
  }
  if (cnt) atomicAdd(&s_cnt, cnt);
  __syncthreads();
  // ---- unreduced diagonal blocks of order > nmin: (start, end) pairs, lowest first ----
  // start[k] = last position j <= k with H1[j, j-1] == 0 (or 0): every thread takes a contiguous
  // chunk, a scan over the threads carries the last zero across the chunks
  __shared__ int s_carry[1024];
  __shared__ int s_nb, s_blo[MS_SCAN_CAND], s_bhi[MS_SCAN_CAND];
  if (tid == 0) s_nb = 0;
  const int chunk = (n + nt - 1) / nt;
  const int k0 = min(n, tid * chunk), k1 = min(n, k0 + chunk);
  int lastz = -1;
  for (int k = k0; k < k1; k++)
    if (k == 0 || !nz[k]) lastz = k;
  s_carry[tid] = lastz;
  __syncthreads();
  for (int o = 1; o < nt; o <<= 1) {
    const int v = (tid >= o) ? s_carry[tid - o] : -1;
    __syncthreads();
    if (v > s_carry[tid]) s_carry[tid] = v;
    __syncthreads();
  }
  {
    int start = (tid > 0) ? s_carry[tid - 1] : 0;
    for (int k = k0; k < k1; k++) {
      if (k == 0 || !nz[k]) start = k;
      const bool end = (k == n - 1) || !nz[k + 1];
      if (end && k - start + 1 > nmin) {
        const int idx = atomicAdd(&s_nb, 1);
        if (idx < MS_SCAN_CAND) { s_blo[idx] = start; s_bhi[idx] = k; }
      }
    }
  }
  __syncthreads();
  if (tid == 0) {
    // lowest blocks first (candidates beyond MS_SCAN_CAND are dropped; later scans find them)
    const int nbk = min(s_nb, MS_SCAN_CAND);
    for (int a = 1; a < nbk; a++) {
      const int lo = s_blo[a], hi = s_bhi[a];
      int b = a - 1;
      while (b >= 0 && s_bhi[b] < hi) { s_blo[b + 1] = s_blo[b]; s_bhi[b + 1] = s_bhi[b]; b--; }
      s_blo[b + 1] = lo; s_bhi[b + 1] = hi;
    }
    const int nout = min(nbk, MS_MAXBLK);
    ctl[0] = (nbk > 0) ? s_blo[0] : 0;
    ctl[1] = (nbk > 0) ? s_bhi[0] : -1;
    ctl[2] = (nbk == 0) ? 1 : 0;
    ctl[3] = s_cnt;
    ctl[5] = nout;
    for (int a = 0; a < nout; a++) { ctl[6 + 2 * a] = s_blo[a]; ctl[7 + 2 * a] = s_bhi[a]; }
    __threadfence();
    *(volatile int*)(ctl + 4) = seq;
    if (prof) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
      ((volatile unsigned long long*)prof)[15] = now;
    }
  }
}

__global__ void __launch_bounds__(1024) ms_scan_kernel(double* H1, int n, int nmin, int* ctl, int seq,
                                                       const WinDesc* wins, int nwin, int W, int D,
                                                       long long* prof) {
  ms_scan_body(H1, n, nmin, ctl, seq, wins, nwin, W, D, prof, reinterpret_cast<unsigned char*>(ms_smem));
}

// debug: stamps the device clock (launch-gap experiments)
__global__ void ms_stamp_kernel(long long* prof, int slot) {
  if (threadIdx.x == 0 && prof) {
    unsigned long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    const unsigned long long last = ((volatile unsigned long long*)prof)[15];
    if (last != 0 && now > last) atomicAdd((unsigned long long*)&prof[slot], now - last);
    ((volatile unsigned long long*)prof)[15] = now;
  }
}

// ------------------------------------------------------------------------------------------
// In-place application of the window factors on the FP64 tensor cores.
//   phase 0: left   H_j[s:s+wl, c_lo:c_hi)  <- U_j' * (same)       tiles of 64 columns
//            and    Z_j[:, s:s+wl)          <- (same) * U_j          tiles of 64 rows
//   phase 1: right  H_jm[r_lo:s, s:s+wl)    <- (same) * U_j,  jm = j-1 (cyclic)
// A CTA reads its whole tile and U_j into shared memory before it writes anything, and tiles of
// one launch are disjoint, so the update is in place without workspace.  (The two phases touch
// the same off-diagonal blocks from different sides, hence two launches.)
// 8 warps as 2 x 4, warp tile 32 x 16 = 4 x 2 DMMA m8n8k4 tiles; operands are kept in their
// natural column-major layout with leading dimension 68 (= 4 mod 16): both fragment patterns
// (8 rows x 4 k and 4 k x 8 columns per half-warp) are then bank-conflict free.
// ------------------------------------------------------------------------------------------
constexpr int AP_T = 64;    // tile extent along the long dimension
constexpr int AP_LD = 68;
constexpr int AP_SMEM = 3 * 64 * AP_LD * 8;  // U_j and two tile buffers

struct ApplyParams {
  int n, p, W, wantT, wantZ, phase, nwin;
  int tpb;  // tiles per CTA (consecutive tiles of one item: U_j is staged once)
  int part;  // 0 all tiles, 1 the tiles next to the windows, 2 the others (see the kernel)
  // Deflation scan fused into the tail of the last update kernel of a round: the CTA that
  // finishes last runs it (a stand-alone one-CTA kernel leaves the GPU idle and was measured to
  // delay the next launch by ~120 us).
  int do_scan, scan_nmin, scan_seq, scan_D;
  int* scan_ctl;
  unsigned int* scan_ticket;  // zero on entry; reset by the scan
  long long* prof;
  double* H[MS_MAXP];
  double* Z[MS_MAXP];
  const double* U;  // U_j of the window at s: wl x wl, leading dimension W, at U + ((j-1) n + s) W
  const WinDesc* wins;
};

// 8-byte asynchronous global -> shared copy (LDGSTS); nbytes = 0 writes zeros without reading.
__device__ __forceinline__ void ms_cp_async8(double* sdst, const double* gsrc, int nbytes) {
  const unsigned sa = (unsigned)__cvta_generic_to_shared(sdst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa), "l"(gsrc), "r"(nbytes) : "memory");
}
__device__ __forceinline__ void ms_cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void ms_cp_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Bulk asynchronous copies (the TMA engine, no LSU instructions per element) completing on an
// mbarrier.  One copy = one contiguous run of a column; addresses and sizes are multiples of 16.
__device__ __forceinline__ unsigned ms_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ms_mbar_init(unsigned long long* b, int cnt) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ms_smem_u32(b)), "r"(cnt) : "memory");
}
__device__ __forceinline__ void ms_mbar_expect_tx(unsigned long long* b, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ms_smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ms_mbar_wait(unsigned long long* b, unsigned parity) {
  asm volatile(
      "{\n.reg .pred p;\nMS_WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MS_WAIT_DONE;\nbra MS_WAIT_LOOP;\nMS_WAIT_DONE:\n}\n" ::"r"(ms_smem_u32(b)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void ms_bulk_g2s(double* sdst, const double* gsrc, unsigned bytes, unsigned long long* b) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   ms_smem_u32(sdst)),
               "l"(gsrc), "r"(bytes), "r"(ms_smem_u32(b))
               : "memory");
}

// Software pipeline per CTA: U_j and the tiles are brought in asynchronously; while tile t is
// multiplied and stored, tile t+1 is already in flight into the other buffer (one CTA barrier per
// tile).  Tiles whose columns are 16-byte aligned runs (the normal case: even n, window start and
// length) come in as bulk copies, one per column, signalled on an mbarrier; anything else falls
// back to 8-byte cp.async.  Results go from the accumulators straight to global memory.
//
// part: 0 = every tile; 1 = only the tiles near the window (the 128 columns right of it for the
// row update, the 64 rows above it for the column update); 2 = the others.  The driver runs part 2
// of round r on a second stream concurrently with the chase of round r+1 (psd_ms.cu,
// CudaBackend::round, explains why that is safe and why the near part has this shape).
__global__ void __launch_bounds__(256, 2) ms_apply_kernel(ApplyParams P) {
  double* Us = ms_smem;               // U(k, c) at Us[c * AP_LD + k]
  double* Xb[2] = {ms_smem + 64 * AP_LD, ms_smem + 2 * 64 * AP_LD};  // X(r, c) at X[c * AP_LD + r]
  __shared__ unsigned long long bar[2], bar_u;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = P.n, p = P.p;
  // item -> (window, factor, kind)
  const int kinds = (P.phase == 0) ? 2 : 1;
  int it = blockIdx.y;
  const int w = it / (p * kinds);
  it -= w * p * kinds;
  const int j = it / kinds + 1;
  const int kind = (P.phase == 0) ? (it % kinds == 0 ? 0 : 2) : 1;  // 0 left, 1 right, 2 Z
  const WinDesc d = P.wins[w];
  const int s = d.s, wl = d.wl;
  double* X;
  int lo, hi;  // extent of the long dimension
  if (kind == 0) {
    X = P.H[j - 1];
    lo = s + wl;
    hi = P.wantT ? n : d.ihi + 1;
  } else if (kind == 1) {
    X = P.H[(j == 1) ? p - 1 : j - 2];
    lo = P.wantT ? 0 : d.ilo;
    hi = s;
  } else {
    X = P.Z[j - 1];
    lo = 0;
    hi = P.wantZ ? n : 0;
  }
  // Tiles of 64 along the long dimension: counted from lo upwards, for the column update from the
  // window (hi = s) upwards, so that tile 0 is always the one next to the window.
  const int nt = (hi > lo) ? (hi - lo + AP_T - 1) / AP_T : 0;
  int ka = 0, kb = nt;  // this launch's tiles of the item
  if (P.part != 0) {
    const int nnear = (kind == 0) ? min(2, nt) : (kind == 1) ? min(1, nt) : 0;
    if (P.part == 1) kb = nnear;
    else ka = nnear;
  }
  auto tile_at = [&](int k, int& t0, int& tl) {
    if (kind == 1) {
      t0 = max(lo, hi - AP_T * (k + 1));
      tl = hi - AP_T * k - t0;
    } else {
      t0 = lo + AP_T * k;
      tl = min(AP_T, hi - t0);
    }
  };
  const int kfirst = ka + blockIdx.x * P.tpb;
  const bool has_work = kfirst < kb && !d.idle;
  if (has_work) {
  const double* Ug = P.U + (size_t)(j - 1) * n * P.W + (size_t)s * P.W;
  // bulk copies need 16-byte aligned runs
  const bool al = ((n | s | wl) & 1) == 0 && ((reinterpret_cast<size_t>(X) | reinterpret_cast<size_t>(P.U)) & 15) == 0;
  if (al) {
    if (tid == 0) { ms_mbar_init(&bar[0], 1); ms_mbar_init(&bar[1], 1); ms_mbar_init(&bar_u, 1); }
    // the padding (rows / columns wl .. 63) is never written by the bulk copies: zero it once
    for (int e = tid; e < 3 * 64 * AP_LD; e += 256) ms_smem[e] = 0.0;
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
  }
  // element (r, cc) of the 64 x 64 staging tile <-> global address, by kind:
  //   left:      rows s .. s+wl-1 (r), columns t0 .. t0+tl-1 (cc)
  //   right / Z: rows t0 .. t0+tl-1 (r), columns s .. s+wl-1 (cc)
  // returns whether the tile went through the bulk path
  auto fetch = [&](double* dst, int t0, int tl, int buf) -> bool {
    if (al && ((t0 | tl) & 1) == 0) {
      const int ncol = (kind == 0) ? tl : wl, len = (kind == 0) ? wl : tl;
      if (tid == 0) ms_mbar_expect_tx(&bar[buf], (unsigned)(ncol * len * 8));
      if (tid < ncol) {
        const double* g = (kind == 0) ? X + s + (size_t)(t0 + tid) * n : X + t0 + (size_t)(s + tid) * n;
        ms_bulk_g2s(dst + tid * AP_LD, g, (unsigned)(len * 8), &bar[buf]);
      }
      return true;
    }
#pragma unroll 4
    for (int i = 0; i < 16; i++) {
      const int e = tid + 256 * i;
      const int r = e & 63, cc = e >> 6;
      bool in;
      const double* g;
      if (kind == 0) {
        in = (r < wl && cc < tl);
        g = X + (s + r) + (size_t)(t0 + cc) * n;
      } else {
        in = (r < tl && cc < wl);
        g = X + (t0 + r) + (size_t)(s + cc) * n;
      }
      ms_cp_async8(dst + cc * AP_LD + r, in ? g : X, in ? 8 : 0);
    }
    ms_cp_commit();
    return false;
  };
  // ---- stage U (wl x wl, zero padded to 64 x 64) and the first tile ----
  unsigned long long* ubar = nullptr;
  if (al) {
    if (tid == 0) ms_mbar_expect_tx(&bar_u, (unsigned)(wl * wl * 8));
    if (tid >= 64 && tid < 64 + wl) ms_bulk_g2s(Us + (tid - 64) * AP_LD, Ug + (size_t)(tid - 64) * P.W, (unsigned)(wl * 8), &bar_u);
    ubar = &bar_u;
  } else {
#pragma unroll 4
    for (int i = 0; i < 16; i++) {
      const int e = tid + 256 * i;
      const int r = e & 63, cc = e >> 6;
      const bool in = (r < wl && cc < wl);
      ms_cp_async8(Us + cc * AP_LD + r, in ? Ug + r + (size_t)cc * P.W : Ug, in ? 8 : 0);
    }
  }
  int t0, tl;
  tile_at(kfirst, t0, tl);
  unsigned par = 0;       // phase parity of the two tile barriers
  unsigned in_bulk = 0;   // bit b: the tile in buffer b came through the bulk path
  if (fetch(Xb[0], t0, tl, 0)) in_bulk |= 1u;
  const int gq = lane >> 2, tq = lane & 3;
  const int kmax = (wl + 3) & ~3;
  // Warp tiles: the 8 x 8 fragments that lie entirely outside the window order wl are skipped, and
  // the split over the warps is chosen so that the two warps of an SM sub-partition (w and w + 4)
  // share that saving: left: 32 window rows x 16 columns, the row half from bit 2 of the warp;
  // right / Z: 16 rows x 32 window columns, the column half from bit 2.
  const int wh = warp >> 2, wq = warp & 3;
  for (int tt = 0; tt < P.tpb; tt++) {
    const int cur = tt & 1;
    double* Xs = Xb[cur];
    ms_cp_wait_all();
    if ((in_bulk >> cur) & 1u) {
      ms_mbar_wait(&bar[cur], (par >> cur) & 1u);
      par ^= 1u << cur;
      in_bulk &= ~(1u << cur);
    }
    if (ubar) {
      ms_mbar_wait(ubar, 0);
      ubar = nullptr;
    }
    __syncthreads();  // tile tt (and U) have landed; every warp is done with the other buffer
    const bool more = (tt + 1 < P.tpb) && (kfirst + tt + 1 < kb);
    int t0n = 0, tln = 0;
    if (more) {
      tile_at(kfirst + tt + 1, t0n, tln);
      // in flight during the multiplication and the store
      if (fetch(Xb[cur ^ 1], t0n, tln, cur ^ 1)) in_bulk |= 1u << (cur ^ 1);
    }
    // ---- C = U' X (left)  or  C = X U (right, Z): 64 x 64 x wl; results go straight from the
    // accumulators to the tile's place in global memory (every element of the tile was read into
    // shared memory before; a lane holds C(row gq, columns 2 tq, 2 tq + 1) of each 8 x 8
    // fragment, so 8 lanes write 64 contiguous bytes) ----
    if (kind == 0) {
      // A(m, k) = U(k, m) = Us[m * LD + k];  B(k, nn) = X(k, nn) = Xs[nn * LD + k]
      double acc[4][2][2];
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int q = 0; q < 2; q++) acc[i][q][0] = acc[i][q][1] = 0.0;
      const int mi = min(4, (wl - wh * 32 + 7) >> 3);
      const double* ap = Us + (wh * 32 + gq) * AP_LD + tq;
      const double* bp = Xs + (wq * 16 + gq) * AP_LD + tq;
      for (int k0 = 0; k0 < kmax; k0 += 4) {
        double a[4], b[2];
#pragma unroll
        for (int i = 0; i < 4; i++) a[i] = ap[i * 8 * AP_LD + k0];
#pragma unroll
        for (int q = 0; q < 2; q++) b[q] = bp[q * 8 * AP_LD + k0];
#pragma unroll
        for (int i = 0; i < 4; i++)
          if (i < mi) {
#pragma unroll
            for (int q = 0; q < 2; q++) ms_dmma(acc[i][q][0], acc[i][q][1], a[i], b[q]);
          }
      }
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int q = 0; q < 2; q++)
#pragma unroll
          for (int e = 0; e < 2; e++) {
            const int m = wh * 32 + i * 8 + gq;
            const int nn = wq * 16 + q * 8 + 2 * tq + e;
            if (m < wl && nn < tl) X[(s + m) + (size_t)(t0 + nn) * n] = acc[i][q][e];
          }
    } else {
      // A(m, k) = X(m, k) = Xs[k * LD + m];  B(k, nn) = U(k, nn) = Us[nn * LD + k]
      double acc[2][4][2];
#pragma unroll
      for (int i = 0; i < 2; i++)
#pragma unroll
        for (int q = 0; q < 4; q++) acc[i][q][0] = acc[i][q][1] = 0.0;
      const int qi = min(4, (wl - wh * 32 + 7) >> 3);
      const double* ap = Xs + tq * AP_LD + wq * 16 + gq;
      const double* bp = Us + (wh * 32 + gq) * AP_LD + tq;
      for (int k0 = 0; k0 < kmax; k0 += 4) {
        double a[2], b[4];
#pragma unroll
        for (int i = 0; i < 2; i++) a[i] = ap[k0 * AP_LD + i * 8];
#pragma unroll
        for (int q = 0; q < 4; q++) b[q] = bp[q * 8 * AP_LD + k0];
#pragma unroll
        for (int q = 0; q < 4; q++)
          if (q < qi) {
#pragma unroll
            for (int i = 0; i < 2; i++) ms_dmma(acc[i][q][0], acc[i][q][1], a[i], b[q]);
          }
      }
#pragma unroll
      for (int i = 0; i < 2; i++)
#pragma unroll
        for (int q = 0; q < 4; q++)
#pragma unroll
          for (int e = 0; e < 2; e++) {
            const int m = wq * 16 + i * 8 + gq;
            const int nn = wh * 32 + q * 8 + 2 * tq + e;
            if (m < tl && nn < wl) X[(t0 + m) + (size_t)(s + nn) * n] = acc[i][q][e];
          }
    }
    if (!more) break;
    t0 = t0n;
    tl = tln;
  }
  }  // has_work
  if (P.do_scan) {
    // last CTA of the grid: every update of the round is complete and visible
    __shared__ unsigned int s_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(P.scan_ticket, 1u) == gridDim.x * gridDim.y - 1) ? 1u : 0u;
    __syncthreads();
    if (s_last) {
      __threadfence();
      ms_scan_body(P.H[0], n, P.scan_nmin, P.scan_ctl, P.scan_seq, P.wins, P.nwin, P.W, P.scan_D, P.prof,
                   reinterpret_cast<unsigned char*>(ms_smem));
      if (tid == 0) *P.scan_ticket = 0;
    }
  }
}

// ------------------------------------------------------------------------------------------
// Shifts: eigenvalues of the trailing nsw x nsw block of the active block, computed by the
// reference algorithm itself (periodic_qr_cta, eigenvalues only) on a copy in shared memory.
// Output: pairs[q] = (re1, im1, re2, im2); ctl[4] = number of pairs.
// `perturb` != 0 spreads the shifts deterministically (exceptional shifts after stagnation).
// ------------------------------------------------------------------------------------------
struct ShiftParams {
  int p, m;            // the snapshot holds the m x m trailing blocks, [p][m * m] column-major
  const double* snap;
  double* pairs;       // this set's pair buffer
  int* state;          // shift_state of ChaseParams
  int slot, seq;
  int lo;              // first row of the block the set is computed from
  double perturb;
};

// Copy of the trailing blocks (rows / columns lo .. lo+m-1 of every factor) taken on the main
// stream, so that the shift computation on a side stream sees one consistent state.
struct SnapParams {
  int n, p, lo, m;
  const double* H[MS_MAXP];
  double* snap;
  int* seq_word;  // the slot's sequence number: cleared here (main stream), so that no window picks
                  // the slot while its pairs are being rewritten
};

__global__ void ms_snapshot_kernel(SnapParams P) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *(volatile int*)P.seq_word = 0;
  const int m = P.m, total = P.p * m * m;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int j = e / (m * m), rem = e - j * m * m;
    const int r = rem % m, cc = rem / m;
    const int keep = (j == 0) ? 1 : 0;
    P.snap[e] = (r > cc + keep) ? 0.0 : P.H[j][(P.lo + r) + (size_t)(P.lo + cc) * P.n];
  }
}

__global__ void __launch_bounds__(256) ms_shifts_kernel(ShiftParams P) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const int m = P.m, p = P.p;
  const int ld = (m % 2 == 0) ? m + 1 : m;
  double* small = ms_smem;
  double* mats = ms_smem + ((rp_small_doubles(m, p) + 1) & ~1LL);
  RCtx c;
  c.n = m; c.p = p; c.tid = tid; c.nt = nt;
  c.hdiag = small;
  c.hsub = c.hdiag + (m + 2);
  c.hsup = c.hsub + (m + 2);
  c.t0 = c.hsup + (m + 2);
  c.t1 = c.t0 + (m + 2);
  c.t2 = c.t1 + (m + 2);
  c.lre = c.t2 + (m + 2);
  c.lim = c.lre + (m + 2);
  c.hnorms = c.lim + (m + 2);
  c.ldh = ld; c.ldz = ld;
  c.H = mats; c.hs = (long long)ld * m;
  c.Z = nullptr; c.zs = 0;
  c.zmap_left = false;
  for (int j = 1; j <= p; j++) {
    const double* src = P.snap + (size_t)(j - 1) * m * m;
    double* dst = c.Hp(j);
    for (int e = tid; e < m * m; e += nt) {
      const int r = e % m, cc = e / m;
      dst[r + (size_t)cc * ld] = src[e];
    }
  }
  __syncthreads();
  int niter = 0;
  const int info = periodic_qr_cta(c, false, false, 30, &niter);
  __syncthreads();
  if (tid == 0) {
    const int np = pair_shifts(c.lre + 1, c.lim + 1, info, m, P.perturb, P.pairs);
    P.state[MS_SS_NP + P.slot] = np;
    P.state[MS_SS_LO + P.slot] = P.lo;
    __threadfence();
    if (np > 0) *(volatile int*)(P.state + MS_SS_SEQ + P.slot) = P.seq;  // publish: this slot holds a complete set
  }
}

// ------------------------------------------------------------------------------------------
// Final stage.  ms_blocklist_kernel: diagonal blocks of H_1 (maximal runs of non-zero
// subdiagonal entries).  1 x 1 blocks get their eigenvalue at once; blocks of order >= 2 are
// listed as WinDesc {s, wl} (ctl[5] = count) for ms_blocks_kernel and the apply kernel.
// ------------------------------------------------------------------------------------------
struct BlockParams {
  int n, p, W, wantT, wantZ, maxitfac;
  double* H[MS_MAXP];
  double* U;
  double* eig;  // [n][2]
  int* info;    // one int (this problem), atomicMax of the failing level
  WinDesc* list;
  int* ctl;
};

__global__ void __launch_bounds__(1024) ms_blocklist_kernel(BlockParams P) {
  const int n = P.n, p = P.p;
  const int tid = threadIdx.x, nt = blockDim.x;
  const double* H1 = P.H[0];
  __shared__ int s_cnt;
  if (tid == 0) s_cnt = 0;
  __syncthreads();
  for (int k = tid; k < n; k += nt) {
    const bool start = (k == 0) || (H1[k + (size_t)(k - 1) * n] == 0.0);
    if (!start) continue;
    int e = k;
    while (e + 1 < n && H1[(e + 1) + (size_t)e * n] != 0.0) e++;
    const int m = e - k + 1;
    if (m == 1) {
      double l = 1.0;
      for (int j = 0; j < p; j++) l *= P.H[j][k + (size_t)k * n];
      P.eig[2 * k] = l;
      P.eig[2 * k + 1] = 0.0;
    } else {
      const int slot = atomicAdd(&s_cnt, 1);
      WinDesc d;
      d.s = k; d.wl = m; d.kbase = 0; d.nbul = 0; d.T = 0; d.ilo = k; d.ihi = e; d.pair0 = 0; d.npairs = 1; d.intro = 0;
      d.idle = 0;
      P.list[slot] = d;
    }
  }
  __syncthreads();
  if (tid == 0) P.ctl[5] = s_cnt;
}

// One CTA per listed block (grid-stride): stage the block of every factor (and an identity for
// the local Schur vectors) in shared memory, run the reference iteration with its 2 x 2
// standardisation (periodic_qr_cta), write the block and V_j (as U_j of this "window") back.
__global__ void __launch_bounds__(256) ms_blocks_kernel(BlockParams P, int nblocks) {
  const int tid = threadIdx.x, nt = blockDim.x;
  const int p = P.p, n = P.n;
  for (int bi = blockIdx.x; bi < nblocks; bi += gridDim.x) {
    const WinDesc d = P.list[bi];
    const int m = d.wl, s = d.s;
    const int ld = (m % 2 == 0) ? m + 1 : m;
    double* small = ms_smem;
    double* mats = ms_smem + ((rp_small_doubles(m, p) + 1) & ~1LL);
    const bool vec = P.wantT || P.wantZ;
    RCtx c;
    c.n = m; c.p = p; c.tid = tid; c.nt = nt;
    c.hdiag = small;
    c.hsub = c.hdiag + (m + 2);
    c.hsup = c.hsub + (m + 2);
    c.t0 = c.hsup + (m + 2);
    c.t1 = c.t0 + (m + 2);
    c.t2 = c.t1 + (m + 2);
    c.lre = c.t2 + (m + 2);
    c.lim = c.lre + (m + 2);
    c.hnorms = c.lim + (m + 2);
    c.ldh = ld; c.ldz = ld;
    c.H = mats; c.hs = (long long)ld * m;
    c.Z = mats + (size_t)p * ld * m; c.zs = (long long)ld * m;
    c.zmap_left = false;
    for (int j = 1; j <= p; j++) {
      const double* src = P.H[j - 1] + s + (size_t)s * n;
      double* dst = c.Hp(j);
      double* z = c.Zp(j);
      const int keep = (j == 1) ? 1 : 0;
      for (int e = tid; e < m * m; e += nt) {
        const int r = e % m, cc = e / m;
        dst[r + (size_t)cc * ld] = (r > cc + keep) ? 0.0 : src[r + (size_t)cc * n];
        if (vec) z[r + (size_t)cc * ld] = (r == cc) ? 1.0 : 0.0;
      }
    }
    __syncthreads();
    int niter = 0;
    const int info = periodic_qr_cta(c, vec, vec, P.maxitfac, &niter);
    __syncthreads();
    for (int k = tid; k < m; k += nt) {
      P.eig[2 * (s + k)] = c.lre[k + 1];
      P.eig[2 * (s + k) + 1] = c.lim[k + 1];
    }
    if (tid == 0 && info != 0) atomicMax(P.info, s + info);
    if (vec) {
      for (int j = 1; j <= p; j++) {
        double* dst = P.H[j - 1] + s + (size_t)s * n;
        const double* src = c.Hp(j);
        const double* z = c.Zp(j);
        double* ud = P.U + (size_t)(j - 1) * n * P.W + (size_t)s * P.W;
        for (int e = tid; e < m * m; e += nt) {
          const int r = e % m, cc = e / m;
          dst[r + (size_t)cc * n] = src[r + (size_t)cc * ld];
          ud[r + (size_t)cc * P.W] = z[r + (size_t)cc * ld];
        }
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------
// Power-of-two normalisation of the factors (the large-N path forms sums of squares and
// products of entries; the reference protects these with scaled sums, householder.jl:5-24,
// 80-100).  sc[j] = 2^-e_j with max |A_j| * sc[j] in [0.5, 1); sc[p + j] = 2^e_j; expo[0] = sum e_j.
// ------------------------------------------------------------------------------------------
__global__ void ms_maxabs_kernel(const double* A, long long count, unsigned long long* out) {
  double m = 0.0;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x) {
    const double v = fabs(A[e]);
    if (v == v) m = fmax(m, v);
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0 && m > 0.0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

__global__ void ms_scales_kernel(const unsigned long long* mx, int p, double* sc, int* expo) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    int tot = 0;
    for (int j = 0; j < p; j++) {
      const double m = __longlong_as_double((long long)mx[j]);
      int e = 0;
      if (m > 0.0 && m < 1.7e308) (void)frexp(m, &e);
      if (e < -1000) e = -1000;  // subnormal maxima: 2^-e itself would overflow
      sc[j] = scalbn(1.0, -e);
      sc[p + j] = scalbn(1.0, e);
      tot += e;
    }
    expo[0] = tot;
  }
}

__global__ void ms_scale_kernel(double* A, long long count, const double* sc) {
  const double s = *sc;
  if (s == 1.0) return;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x)
    A[e] *= s;
}

__global__ void ms_scale_eig_kernel(double* eig, int n, const int* expo) {
  const int e = expo[0];
  if (e == 0) return;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < 2 * n; k += gridDim.x * blockDim.x)
    eig[k] = scalbn(eig[k], e);
}

}  // namespace ms
}  // namespace psd
