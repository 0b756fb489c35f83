// C ABI of the B200 periodic Schur library (see include/psd_b200.h for the contract).
//
// Host side: a handle owns, per device, a small pool of "slots" (stream + device buffers +
// pinned staging).  A batched host call shards the batch into one contiguous range per
// device (one host thread each, no inter-device traffic), cuts each range into chunks and
// round-robins the chunks over the slots so that H2D of chunk c+1, the kernel of chunk c and
// D2H of chunk c-1 overlap on different streams.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <initializer_list>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/psd_b200.h"
#include "psd_real_kernel.cuh"
#include "psd_checkpsd.cuh"
#include "psd_real_hess32.cuh"
#include "psd_cplx_qz.cuh"
#include "psd_rowhess.cuh"
#include "psd_dgemm.cuh"
#include "psd_large_hess.cuh"
#include "psd_ms.h"
#include "psd_rng.cuh"

namespace {

thread_local std::string g_err;

// Experiment switches (PSD_* environment variables) exist only in builds made with
// -DPSD_DEBUG_ENV; the product library never reads the environment.
inline const char* dbg_env(const char* name) {
#ifdef PSD_DEBUG_ENV
  return getenv(name);
#else
  (void)name;
  return nullptr;
#endif
}

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define PSD_CUDA(call)                                                                     \
  do {                                                                                     \
    cudaError_t e__ = (call);                                                              \
    if (e__ != cudaSuccess)                                                                \
      return fail(PSD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));      \
  } while (0)

constexpr int kSlotsPerDevice = 3;

// Roles of the pipeline buffers of a batched host call: the factors (A in, T out), Z, the
// eigenvalues (real: eig in kVal0; generalized: alpha, beta, alphascale), info, iteration counts.
enum Role { kFactors, kZ, kVal0, kVal1, kVal2, kInfo, kIters, kRoles };

struct Slot {
  cudaStream_t stream = nullptr;
  // pipeline buffers by role: device, and pinned staging (only used when the caller's buffers are
  // pageable); the pipeline copies these out, so no launch function uses them as scratch
  void* dBuf[kRoles] = {};
  size_t dCap[kRoles] = {};
  void* hBuf[kRoles] = {};
  size_t hCap[kRoles] = {};
  double* dArg[3] = {};  // operands of the single-slot entry points (rphess_packed, rowwise, dgemm)
  size_t capArg[3] = {};
  unsigned long long* dCounter = nullptr;  // [2]: reduction kernel, QR kernel
  double* dScratch = nullptr;
  size_t capScratch = 0;
  double* dPacked = nullptr;  // packed Hessenberg-triangular factors between the two kernels
  size_t capPacked = 0;
  double* dPk[8] = {nullptr};  // packed leading parts handed to the later occupancy phases
  size_t capPk[8] = {0};
  unsigned long long* dPhaseCtr = nullptr;  // work counters of the phase launches
  unsigned char* dS = nullptr;  // generalized paths: the signature
  size_t capS = 0;
  psd::ms::Workspace* ms = nullptr;  // large-N multishift iteration (psd_ms.cu)
  void* dTeam[3] = {};  // team iteration scratch: alpha, beta, alphascale
  size_t capTeam[3] = {};
  // iteration counts (psd_set_iters_output) of the chunk being enqueued, read by the launch
  // functions (nullptr: not wanted)
  int32_t* curIters = nullptr;
  double* curTau = nullptr;  // psd_rphess_packed_batched: device tau of the chunk being enqueued
  long long* dProf = nullptr;        // PSD_PANEL_PROF cycle counters (debug builds)
};

struct Device {
  int ordinal = 0;
  int sm_count = 0;
  Slot slots[kSlotsPerDevice];
  Slot user;  // counter/scratch for *_dev entry points running on caller streams
  cudaEvent_t userDone = nullptr;  // last *_dev call on this device (they share `user`)
};

}  // namespace

struct KernelTimer {
  cudaEvent_t e0, e1;
  int kind;     // 0 = reduction kernel, 1 = QR/QZ iteration kernel, 2 = large-N panel, 3 = large-N GEMMs
  int ordinal;  // device the events belong to
};

struct psd_handle_s {
  std::vector<Device> devs;
  std::mutex mu;
  int64_t stats[8] = {0};
  bool profiling = false;           // psd_set_profiling
  std::vector<KernelTimer> timers;  // pending event pairs (resolved by psd_kernel_times)
  double gemm_flops = 0.0;          // FP64 GEMM flops issued by the large-N reduction since then
  double extra_launches = 0.0;      // kernel launches covered by a timer that brackets several
  psd::ms::Result ms_last;          // counters of the most recent large-N iteration
  int32_t* iters_host = nullptr;    // psd_set_iters_output
  std::mutex tmu;
};

namespace {

template <class T>
int ensure_dev(T*& ptr, size_t& cap, size_t bytes) {
  if (bytes <= cap) return PSD_OK;
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cap = 0;
  PSD_CUDA(cudaMalloc((void**)&ptr, bytes));
  cap = bytes;
  return PSD_OK;
}
template <class T>
int ensure_pinned(T*& ptr, size_t& cap, size_t bytes) {
  if (bytes <= cap) return PSD_OK;
  if (ptr) cudaFreeHost(ptr);
  ptr = nullptr;
  cap = 0;
  PSD_CUDA(cudaHostAlloc((void**)&ptr, bytes, cudaHostAllocDefault));
  cap = bytes;
  return PSD_OK;
}

bool is_pinned(const void* p) {
  if (!p) return true;
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// The single-slot entry points run on slot 0 of the handle's first device: make that device
// current and wait until the slot's stream is idle.
int use_slot0(psd_handle_s* h) {
  Device& dev = h->devs[0];
  PSD_CUDA(cudaSetDevice(dev.ordinal));
  Slot& s = dev.slots[0];
  if (!s.stream) PSD_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
  PSD_CUDA(cudaStreamSynchronize(s.stream));
  return PSD_OK;
}

// Bracket a kernel launch with CUDA events on its stream when profiling is enabled.
struct ScopedKernelTimer {
  psd_handle_s* h;
  cudaStream_t st;
  KernelTimer t;
  bool on;
  ScopedKernelTimer(psd_handle_s* h_, const Device& dev, cudaStream_t st_, int kind) : h(h_), st(st_) {
    on = h->profiling;
    if (!on) return;
    t.kind = kind;
    t.ordinal = dev.ordinal;
    cudaEventCreate(&t.e0);
    cudaEventCreate(&t.e1);
    cudaEventRecord(t.e0, st);
  }
  ~ScopedKernelTimer() {
    if (!on) return;
    cudaEventRecord(t.e1, st);
    std::lock_guard<std::mutex> lk(h->tmu);
    h->timers.push_back(t);
  }
};

struct RealLaunchPlan {
  int use_smem = 0;
  int ldh = 0;
  int threads = 64;
  size_t smem_bytes = 0;
  int grid = 1;
  bool scratch = false;
};

// Choose staging mode, CTA size and persistent grid for the real kernel.
int plan_real(const Device& dev, int n, int p, long long batch, bool wantZ, RealLaunchPlan& pl) {
  const long long small = psd::rp_small_doubles(n, p);
  const int ldh = (n % 2 == 0) ? n + 1 : n;
  const long long mats = (long long)p * ldh * n * (wantZ ? 2 : 1);
  const size_t need_smem = (size_t)(small + mats) * sizeof(double);
  cudaFuncAttributes fa;
  PSD_CUDA(cudaFuncGetAttributes(&fa, psd::rpschur_kernel));
  int optin = 0;
  PSD_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev.ordinal));
  const size_t max_dyn = (size_t)optin - fa.sharedSizeBytes;
  if (need_smem <= max_dyn) {
    pl.use_smem = 1;
    pl.ldh = ldh;
    pl.smem_bytes = need_smem;
    pl.scratch = false;
  } else {
    pl.use_smem = 0;
    pl.ldh = n;
    if ((size_t)small * sizeof(double) <= 96 * 1024) {
      pl.smem_bytes = (size_t)small * sizeof(double);
      pl.scratch = false;
    } else {
      pl.smem_bytes = 0;
      pl.scratch = true;
    }
  }
  // one row or column per thread for the left, right and Z updates
  int want = n * (wantZ ? 3 : 2);
  int threads = ((want + 31) / 32) * 32;
  threads = std::max(32, std::min(threads, 256));  // 254 registers per thread: 256 threads fill an SM's file
  pl.threads = threads;
  PSD_CUDA(cudaFuncSetAttribute(psd::rpschur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)max_dyn));
  int occ = 0;
  PSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, psd::rpschur_kernel, threads,
                                                         pl.smem_bytes));
  if (occ < 1) return fail(PSD_ERR_UNSUPPORTED, "kernel does not fit on an SM");
  long long g = (long long)occ * dev.sm_count;
  pl.grid = (int)std::max(1LL, std::min(g, batch));
  return PSD_OK;
}

struct RealCall {
  int n, p, left, wantT, wantZ, maxitfac, reduce_only, skip_reduce;
  int z_preset = 0;
};

constexpr int kLargeN = 192;  // from here on the reduction runs blocked on the whole GPU

constexpr long long kEigChunk = 65536;  // problems per (reduction, QR) kernel pair

// Eigenvalue-only fast path for n <= 32: reduction kernel -> packed factors -> one warp per
// problem QR kernel (psd_real_eig32.cuh).
int launch_real_eig32(psd_handle_s* h, Device& dev, Slot& aux, cudaStream_t stream, const RealCall& rc,
                      long long batch, double* dA, double* dEig, int32_t* dInfo) {
  const int n = rc.n, p = rc.p;
  const size_t nn = (size_t)n * n;
  const size_t psize = (size_t)psd::pk_problem_size(n, p);
  long long chunk_max = kEigChunk;
  if (const char* ev = dbg_env("PSD_EIG_CHUNK")) chunk_max = std::max(1LL, atoll(ev));
  const long long chunk = std::min(batch, chunk_max);
  int e = ensure_dev(aux.dPacked, aux.capPacked, (size_t)chunk * psd::pk_problem_stride(n, p) * sizeof(double));
  if (e) return e;
  if (!aux.dCounter) PSD_CUDA(cudaMalloc((void**)&aux.dCounter, 2 * sizeof(unsigned long long)));
  if (!aux.dPhaseCtr) PSD_CUDA(cudaMalloc((void**)&aux.dPhaseCtr, 16 * sizeof(unsigned long long)));
  int optin = 0;
  PSD_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev.ordinal));
  // occupancy phases of the iteration (see rpqr_eig32_kernel_t): orders n, 7n/8, ..., 3n/8
  struct Phase {
    int n, stop, wpb, grid;
    size_t smem;
    void (*kern)(psd::EigParams);
  };
  std::vector<Phase> phases;
  {
    std::vector<int> orders{n};
    if (n >= 24 && !dbg_env("PSD_NO_PHASES"))
      for (int k = 1; k <= 5; k++) orders.push_back(n - k * (n / 8));  // n = 32: 28, 24, 20, 16, 12
    bool special = (n == 32 && p == 8 && !dbg_env("PSD_NO_SPECIAL"));
    if (const char* ev = dbg_env("PSD_PHASES")) {  // experiment: comma-separated decreasing orders after n
      orders.assign(1, n);
      for (const char* c = ev; *c;) {
        int v = atoi(c);
        if (v > 1 && v < orders.back()) orders.push_back(v);
        while (*c && *c != ',') c++;
        if (*c == ',') c++;
      }
    }
    for (size_t k = 0; k < orders.size(); k++) {
      Phase ph;
      ph.n = orders[k];
      ph.stop = (k + 1 < orders.size()) ? orders[k + 1] : 0;
      ph.kern = psd::rpqr_eig32_kernel_t<0, 0>;
      if (special && k == 0) ph.kern = psd::rpqr_eig32_kernel_t<32, 8>;
      int wmax = 8;
      if (k > 0) {
        const char* lr = dbg_env("PSD_LOWREG");
        const int mode = lr ? atoi(lr) : 168;
        if (mode == 168) { ph.kern = psd::rpqr_eig32_kernel_r168; wmax = 3; }
        if (mode == 128) { ph.kern = psd::rpqr_eig32_kernel_r128; wmax = 4; }
      }
      cudaFuncAttributes fa;
      PSD_CUDA(cudaFuncGetAttributes(&fa, ph.kern));
      const size_t max_dyn = (size_t)optin - fa.sharedSizeBytes;
      const size_t pbytes = (size_t)psd::pk_problem_size(ph.n, p) * sizeof(double);
      PSD_CUDA(cudaFuncSetAttribute(ph.kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_dyn));
      // several CTAs per SM only fit with the largest shared-memory carve-out
      PSD_CUDA(cudaFuncSetAttribute(ph.kern, cudaFuncAttributePreferredSharedMemoryCarveout,
                                    (int)cudaSharedmemCarveoutMaxShared));
      // warps per CTA: the split that gives the most resident warps per SM (<= 8 warps per CTA)
      int best_w = 0, best_total = 0;
      for (int w = 1; w <= wmax; w++) {
        if ((size_t)w * pbytes > max_dyn) break;
        int occ = 0;
        PSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, ph.kern, w * 32, (size_t)w * pbytes));
        if (dbg_env("PSD_GEN_PROF")) fprintf(stderr, "[psd eig32 occ] order %d w %d -> %d CTAs/SM\n", ph.n, w, occ);
        if (occ * w > best_total || (occ * w == best_total && w > best_w)) {
          best_total = occ * w;
          best_w = w;
        }
      }
      if (best_w < 1) return fail(PSD_ERR_UNSUPPORTED, "packed problem does not fit in shared memory");
      if (const char* ev = dbg_env("PSD_PHASE_WPB")) {  // experiment: force warps per CTA, oversubscribed grid
        const int w = atoi(ev);
        if (k > 0 && w >= 1 && (size_t)w * pbytes <= max_dyn) {
          best_w = w;
          best_total = w * 4;
        }
      }
      ph.wpb = best_w;
      ph.smem = (size_t)best_w * pbytes;
      ph.grid = (best_total / best_w) * dev.sm_count;
      if (dbg_env("PSD_GEN_PROF"))
        fprintf(stderr, "[psd eig32 phase %zu] order %d stop %d: %d warps/CTA x %d CTAs/SM, %zu B smem/CTA, %d regs\n", k,
                ph.n, ph.stop, best_w, best_total / best_w, ph.smem, fa.numRegs);
      phases.push_back(ph);
    }
    if (phases.size() > 9) return fail(PSD_ERR_BAD_ARG, "too many phases");
    for (size_t k = 1; k < phases.size(); k++)
      if ((e = ensure_dev(aux.dPk[k - 1], aux.capPk[k - 1],
                          (size_t)chunk * psd::pk_problem_stride(phases[k].n, p) * sizeof(double))))
        return e;
  }
  for (long long off = 0; off < batch; off += chunk) {
    const long long nb = std::min(chunk, batch - off);
    PSD_CUDA(cudaMemsetAsync(aux.dCounter, 0, 2 * sizeof(unsigned long long), stream));
    if (rc.skip_reduce) {
      // input already Hessenberg/triangular: CTA kernel only enforces structure and packs
      RealLaunchPlan pl;
      e = plan_real(dev, n, p, nb, false, pl);
      if (e) return e;
      if (!pl.use_smem) return fail(PSD_ERR_UNSUPPORTED, "eig32 path expects shared-memory staging");
      psd::RpschurParams P;
      P.n = n; P.p = p; P.batch = nb;
      P.left = rc.left; P.wantT = 0; P.wantZ = 0; P.maxitfac = 30;
      P.A = dA + (size_t)off * p * nn; P.Z = nullptr; P.eig = nullptr; P.info = nullptr; P.iters = nullptr;
      P.use_smem = pl.use_smem; P.ldh = pl.ldh;
      P.reduce_only = 1; P.skip_reduce = rc.skip_reduce; P.z_preset = 0;
      P.counter = aux.dCounter;
      P.scratch = nullptr; P.scratch_stride = 0;
      P.packed_out = aux.dPacked;
      P.tau = nullptr;
      ScopedKernelTimer tm(h, dev, stream, 0);
      psd::rpschur_kernel<<<pl.grid, pl.threads, pl.smem_bytes, stream>>>(P);
      PSD_CUDA(cudaGetLastError());
    } else {
      psd::Hess32Params R;
      R.n = n; R.p = p; R.batch = nb; R.left = rc.left;
      R.ld = (n % 2 == 0) ? n + 1 : n;
      R.A = dA + (size_t)off * p * nn;
      R.packed_out = aux.dPacked;
      R.counter = aux.dCounter;
      // p >= 2: two warps per problem (rphess_pair32_kernel_t), or, where it is faster, a chain warp
      // that runs the reflector chain up to p-2 steps ahead of two warps applying the left and right
      // updates (rphess_ahead32_kernel_t).  The chain-ahead kernel needs p >= 7 to run far enough
      // ahead (measured slower at p = 3..6), and its 168-register warps must not leave fewer
      // problems resident per SM than the two-warp kernel (measured slower at N = 17, p = 8, where
      // registers hold it to 4 problems per SM against 12).  p = 1 keeps one warp per problem.
      const bool special = n == 32 && p == 8 && !dbg_env("PSD_NO_SPECIAL");
      struct Shape {
        void (*k)(psd::Hess32Params);
        int wpp, wpb, occ;
        size_t smem;
      };
      const size_t staged = (size_t)p * R.ld * n * sizeof(double);
      auto shape = [&](void (*k)(psd::Hess32Params), int wpp, size_t per, Shape& sh) -> int {
        cudaFuncAttributes fh;
        PSD_CUDA(cudaFuncGetAttributes(&fh, k));
        const size_t max_dyn = (size_t)optin - fh.sharedSizeBytes;
        sh.k = k;
        sh.wpp = wpp;
        sh.wpb = (int)std::min<size_t>(std::min(8, fh.maxThreadsPerBlock / (32 * wpp)), max_dyn / per);
        sh.occ = 0;
        if (sh.wpb < 1) return PSD_OK;
        sh.smem = (size_t)sh.wpb * per;
        PSD_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_dyn));
        PSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&sh.occ, k, sh.wpb * wpp * 32, sh.smem));
        return PSD_OK;
      };
      Shape hs;
      if (p == 1) {
        if ((e = shape(special ? psd::rphess_warp32_kernel_t<32, 8> : psd::rphess_warp32_kernel_t<0, 0>, 1, staged, hs)))
          return e;
      } else {
        if ((e = shape(psd::rphess_pair32_kernel_t<0, 0>, 2, staged, hs))) return e;
        if (p >= 7) {
          Shape as;
          if ((e = shape(special ? psd::rphess_ahead32_kernel_t<32, 8> : psd::rphess_ahead32_kernel_t<0, 0>,
                         psd::AHEAD_WARPS, psd::ahead_problem_doubles(n, p, R.ld) * sizeof(double), as)))
            return e;
          if (as.occ > 0 && as.wpb * as.occ >= hs.wpb * hs.occ) hs = as;
        }
      }
      if (hs.occ < 1) return fail(PSD_ERR_UNSUPPORTED, "reduction kernel does not fit on an SM");
      const int wpb1 = hs.wpb, wpp = hs.wpp, occ1 = hs.occ;
      const size_t smem1 = hs.smem;
      void (*hk)(psd::Hess32Params) = hs.k;
      const long long ctas1 = (nb + wpb1 - 1) / wpb1;
      const int grid1 = (int)std::max(1LL, std::min((long long)occ1 * dev.sm_count, ctas1));
      if (dbg_env("PSD_GEN_PROF"))
        fprintf(stderr, "[psd hess32] %d warps/problem, %d problems/CTA x %d CTAs/SM, %zu B smem/CTA\n", wpp, wpb1,
                occ1, smem1);
      {
        ScopedKernelTimer tm(h, dev, stream, 0);
        hk<<<grid1, wpb1 * wpp * 32, smem1, stream>>>(R);
      }
      PSD_CUDA(cudaGetLastError());
    }
    PSD_CUDA(cudaMemsetAsync(aux.dPhaseCtr, 0, 16 * sizeof(unsigned long long), stream));
    {
      ScopedKernelTimer tm(h, dev, stream, 1);  // the phase launches are timed as one iteration
      for (size_t k = 0; k < phases.size(); k++) {
        const Phase& ph = phases[k];
        psd::EigParams Q;
        Q.n = ph.n; Q.p = p; Q.batch = nb; Q.maxitfac = rc.maxitfac > 0 ? rc.maxitfac : 30;
        Q.packed = (k == 0) ? aux.dPacked : aux.dPk[k - 1];
        Q.packed_next = (k + 1 < phases.size()) ? aux.dPk[k] : nullptr;
        Q.n_full = n; Q.stop = ph.stop; Q.first_phase = (k == 0) ? 1 : 0;
        Q.eig = dEig + (size_t)off * 2 * n;
        Q.info = dInfo + off;
        Q.iters = aux.curIters ? aux.curIters + off : nullptr;
        Q.counter = aux.dPhaseCtr + k;
        Q.force_safe = dbg_env("PSD_EIG32_SAFE") ? 1 : 0;
        const long long ctas = (nb + ph.wpb - 1) / ph.wpb;
        const int grid2 = (int)std::max(1LL, std::min((long long)ph.grid, ctas));
        ph.kern<<<grid2, ph.wpb * 32, ph.smem, stream>>>(Q);
      }
    }
    PSD_CUDA(cudaGetLastError());
    {
      std::lock_guard<std::mutex> lk(h->tmu);
      h->extra_launches += (double)(phases.size() - 1);
    }
    __atomic_fetch_add(&h->stats[0], (int64_t)2, __ATOMIC_RELAXED);
  }
  __atomic_fetch_add(&h->stats[1], (int64_t)batch, __ATOMIC_RELAXED);
  return PSD_OK;
}


// Large-N path: blocked periodic Hessenberg-triangular reduction on the whole GPU (one problem at
// a time), then the periodic QR iteration on the reduced factors with Z preset to the Q_j.
int launch_real_large(psd_handle_s* h, Device& dev, Slot& aux, cudaStream_t stream, const RealCall& rc,
                      long long batch, double* dA, double* dZ, double* dEig, int32_t* dInfo);
bool large_feasible(const Device& dev, int n, int p);

// Enqueue the real kernel for `batch` device-resident problems on `stream`.
int launch_real(psd_handle_s* h, Device& dev, Slot& aux, cudaStream_t stream, const RealCall& rc,
                long long batch, double* dA, double* dZ, double* dEig, int32_t* dInfo) {
  if (batch == 0) return PSD_OK;
  RealLaunchPlan pl;
  const bool wantZ = rc.wantZ && dZ;
  if (rc.n >= kLargeN && !rc.skip_reduce && !aux.curTau && !dbg_env("PSD_DISABLE_LARGE") && large_feasible(dev, rc.n, rc.p))
    return launch_real_large(h, dev, aux, stream, rc, batch, dA, dZ, dEig, dInfo);
  if (!rc.wantT && !wantZ && !rc.reduce_only && rc.n <= 32 && rc.p >= 3 && !dbg_env("PSD_DISABLE_EIG32"))
    return launch_real_eig32(h, dev, aux, stream, rc, batch, dA, dEig, dInfo);
  int e = plan_real(dev, rc.n, rc.p, batch, wantZ, pl);
  if (e) return e;
  if (!aux.dCounter) PSD_CUDA(cudaMalloc((void**)&aux.dCounter, 2 * sizeof(unsigned long long)));
  PSD_CUDA(cudaMemsetAsync(aux.dCounter, 0, sizeof(unsigned long long), stream));
  psd::RpschurParams P;
  P.n = rc.n; P.p = rc.p; P.batch = batch;
  P.left = rc.left; P.wantT = rc.wantT; P.wantZ = wantZ ? 1 : 0;
  P.maxitfac = rc.maxitfac > 0 ? rc.maxitfac : 30;
  P.A = dA; P.Z = wantZ ? dZ : nullptr; P.eig = dEig; P.info = dInfo; P.iters = aux.curIters;
  P.use_smem = pl.use_smem; P.ldh = pl.ldh;
  P.reduce_only = rc.reduce_only; P.skip_reduce = rc.skip_reduce; P.z_preset = rc.z_preset;
  P.counter = aux.dCounter;
  P.scratch = nullptr; P.scratch_stride = 0;
  P.packed_out = nullptr;
  P.tau = aux.curTau;
  if (pl.scratch) {
    size_t stride = (size_t)psd::rp_small_doubles(rc.n, rc.p);
    e = ensure_dev(aux.dScratch, aux.capScratch, stride * sizeof(double) * pl.grid);
    if (e) return e;
    P.scratch = aux.dScratch;
    P.scratch_stride = (long long)stride;
  }
  {
    ScopedKernelTimer tm(h, dev, stream, 1);
    psd::rpschur_kernel<<<pl.grid, pl.threads, pl.smem_bytes, stream>>>(P);
  }
  PSD_CUDA(cudaGetLastError());
  __atomic_fetch_add(&h->stats[0], (int64_t)1, __ATOMIC_RELAXED);
  __atomic_fetch_add(&h->stats[pl.use_smem ? 1 : 2], (int64_t)batch, __ATOMIC_RELAXED);
  return PSD_OK;
}


// Feasibility of the blocked large-N reduction on this device (slab scheme of the panel kernel,
// its shared memory, one resident CTA per SM); otherwise the generic CTA kernel takes the problem.
bool large_feasible(const Device& dev, int n, int p) {
  if (p > psd::LH_MAXP) return false;
  const int nb = psd::lh_panel_width(p);
  int R = (n + dev.sm_count - 1) / dev.sm_count;
  R = (R + 3) & ~3;
  if (R > psd::LH_RMAX) return false;
  int optin = 0;
  if (cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev.ordinal) != cudaSuccess) return false;
  const size_t smem = ((size_t)p * nb * nb + n) * sizeof(double);
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, psd::rphess_panel_kernel) != cudaSuccess) return false;
  if (smem + fa.sharedSizeBytes > (size_t)optin) return false;
  if (cudaFuncSetAttribute(psd::rphess_panel_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, psd::rphess_panel_kernel, psd::LH_THREADS, smem) != cudaSuccess || occ < 1) {
    cudaGetLastError();
    return false;
  }
  return true;
}

// Team-mode iteration (one double-shift bulge at a time on the whole GPU): the fallback of the
// large-N path when the multishift iteration does not apply (p > 12) or reports no convergence.
int launch_team_iteration(psd_handle_s* h, Device& dev, Slot& aux, cudaStream_t stream, const RealCall& rc,
                          long long batch, double* dA, double* dZ, double* dEig, int32_t* dInfo) {
  const int n = rc.n, p = rc.p;
  const bool wantZ = rc.wantZ && dZ;
  int e;
  const size_t cnt = (size_t)batch * n;
  if ((e = ensure_dev(aux.dTeam[0], aux.capTeam[0], cnt * 16))) return e;
  if ((e = ensure_dev(aux.dTeam[1], aux.capTeam[1], cnt * 8))) return e;
  if ((e = ensure_dev(aux.dTeam[2], aux.capTeam[2], cnt * 8))) return e;
  psd::GpqzParams<double> P;
  P.n = n; P.p = p; P.batch = batch; P.left = rc.left; P.wantT = rc.wantT; P.wantZ = wantZ ? 1 : 0;
  P.maxitfac = 4 * (rc.maxitfac > 0 ? rc.maxitfac : 30);  // QZ loop counts deflation steps too (rgeneralized.jl:52)
  P.skip_reduce = 1; P.reduce_only = 0;
  P.S = nullptr;
  P.A = dA; P.Z = wantZ ? dZ : nullptr;
  P.alpha = (psd::cplx*)aux.dTeam[0]; P.beta = (double*)aux.dTeam[1]; P.scale = (long long*)aux.dTeam[2];
  P.info = dInfo;
  P.use_smem = 0; P.ldh = n; P.debug = 0; P.counter = nullptr; P.blocked_stage1 = 0; P.windowed_stage2 = 0; P.windowed_qz = 0;
  P.deep = 4;  // team mode: < 1 element pair per thread and factor, one pass instead of p + 1 (N = 1024: 7.1 s -> 5.3 s)
  if (const char* ev = dbg_env("PSD_DEEP_U")) P.deep = atoi(ev);
  auto kern = psd::gpschur_team_kernel<double>;
  size_t smem = (size_t)((psd::cq_small_doubles(n, p) + 1) & ~1LL) * sizeof(double);
  if (!dbg_env("PSD_NO_WINDOWED_QZ")) {
    P.windowed_qz = 1;  // batches of 12 bulge steps between grid barriers instead of two barriers per step
    smem += (size_t)psd::qzw_work_doubles(p, psd::S3_K_TEAM) * sizeof(double);
  }
  PSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int occ = 0;
  PSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, smem));
  if (occ < 1) return fail(PSD_ERR_UNSUPPORTED, "team kernel does not fit on an SM");
  int zp = 1;
  void* args[] = {&P, &zp};
  int ctas = dev.sm_count;
  if (const char* ev = dbg_env("PSD_TEAM_CTAS")) ctas = std::max(1, std::min(atoi(ev), dev.sm_count * occ));
  {
    ScopedKernelTimer tm(h, dev, stream, 1);
    PSD_CUDA(cudaLaunchCooperativeKernel((void*)kern, dim3(ctas), dim3(256), args, smem, stream));
  }
  psd::gvalues_kernel<<<std::min<long long>(1024, (long long)(cnt + 255) / 256), 256, 0, stream>>>(
      (const psd::cplx*)aux.dTeam[0], (const double*)aux.dTeam[1], (const long long*)aux.dTeam[2], dEig, (long long)cnt);
  PSD_CUDA(cudaGetLastError());
  __atomic_fetch_add(&h->stats[0], (int64_t)2, __ATOMIC_RELAXED);
  return PSD_OK;
}

int launch_real_large(psd_handle_s* h, Device& dev, Slot& aux, cudaStream_t stream, const RealCall& rc,
                      long long batch, double* dA, double* dZ, double* dEig, int32_t* dInfo) {
  const int n = rc.n, p = rc.p;
  const size_t nn = (size_t)n * n;
  const bool wantZ = rc.wantZ && dZ;
  int e = ensure_dev(aux.dScratch, aux.capScratch,
                     (psd::lh_work_doubles(n, p) + (size_t)psd::rp_small_doubles(n, p) * 2) * sizeof(double));
  if (e) return e;
  double* work = aux.dScratch + (size_t)psd::rp_small_doubles(n, p) * 2;  // QR scratch lives in front
  if (!aux.ms) aux.ms = psd::ms::ws_create();
  // Exact power-of-two normalisation of every factor (undone on T and the eigenvalues at the end):
  // the blocked reduction forms sums of squares and the iteration products of entries, which the
  // reference protects with scaled sums (householder.jl:5-24, 80-100).
  const bool scaled = p <= psd::ms::kMaxPeriod && !dbg_env("PSD_NO_PRESCALE");
  const bool use_ms = psd::ms::supported(n, p) && !rc.reduce_only && !dbg_env("PSD_DISABLE_MS");
  bool team_needed = false;
  for (long long b = 0; b < batch; b++) {
    double* Ab = dA + (size_t)b * p * nn;
    double* Zb = wantZ ? dZ + (size_t)b * p * nn : nullptr;
    double* Ap[psd::LH_MAXP];
    double* Qp[psd::LH_MAXP];
    for (int j = 1; j <= p; j++) {
      Ap[j - 1] = Ab + (size_t)((rc.left ? (p + 1 - j) : j) - 1) * nn;
      const int s = (rc.left && j > 1) ? (p + 2 - j) : j;
      Qp[j - 1] = Zb ? Zb + (size_t)(s - 1) * nn : nullptr;
    }
    if (scaled) PSD_CUDA(psd::ms::prescale(stream, aux.ms, n, p, Ap));
    double fl = 0.0;
    std::vector<ScopedKernelTimer*> open(4, nullptr);
    auto mark = [&](int kind, int phase) {
      if (phase == 0) {
        open[kind] = new ScopedKernelTimer(h, dev, stream, kind);
      } else {
        delete open[kind];
        open[kind] = nullptr;
      }
    };
    long long* dprof = nullptr;
    if (dbg_env("PSD_PANEL_PROF")) {
      if (!aux.dProf) PSD_CUDA(cudaMalloc((void**)&aux.dProf, 8 * sizeof(long long)));
      PSD_CUDA(cudaMemsetAsync(aux.dProf, 0, 8 * sizeof(long long), stream));
      dprof = aux.dProf;
    }
    cudaError_t ce = psd::rphess_large(stream, dev.sm_count, n, p, Ap, Zb ? Qp : nullptr, work, &fl, mark, dprof);
    if (dprof) {
      long long hp[8];
      PSD_CUDA(cudaMemcpyAsync(hp, dprof, sizeof(hp), cudaMemcpyDeviceToHost, stream));
      PSD_CUDA(cudaStreamSynchronize(stream));
      fprintf(stderr, "[psd panel cycles, CTA 0] s1+s2 %lld | wait S2 %lld | s3 %lld | wait S3 %lld | s4 head+gemv %lld | s4 tail %lld\n",
              hp[0], hp[1], hp[2], hp[3], hp[4], hp[5]);
    }
    for (auto* t : open) delete t;
    if (ce != cudaSuccess) return fail(PSD_ERR_CUDA, std::string("large-N reduction: ") + cudaGetErrorString(ce));
    {
      std::lock_guard<std::mutex> lk(h->tmu);
      h->gemm_flops += fl;
    }
    __atomic_fetch_add(&h->stats[0], (int64_t)((n + 63) / 64) * (1 + 7 * p), __ATOMIC_RELAXED);
    if (rc.reduce_only) {
      if (scaled) PSD_CUDA(psd::ms::postscale(stream, aux.ms, n, p, Ap, 1, nullptr));
      continue;
    }
    if (use_ms) {
      // Small-bulge multishift sweeps in diagonal windows + tensor-core updates (psd_ms.cu).
      PSD_CUDA(cudaMemsetAsync(dInfo + b, 0, sizeof(int32_t), stream));
      psd::ms::Result res;
      {
        ScopedKernelTimer tm(h, dev, stream, 1);
        ce = psd::ms::iterate(stream, dev.sm_count, aux.ms, n, p, Ap, Zb ? Qp : nullptr, rc.wantT, wantZ ? 1 : 0,
                              rc.maxitfac, dEig + (size_t)b * 2 * n, dInfo + b, h->profiling ? 1 : 0, &res);
      }
      if (ce != cudaSuccess) return fail(PSD_ERR_CUDA, std::string("large-N iteration: ") + cudaGetErrorString(ce));
      {
        std::lock_guard<std::mutex> lk(h->tmu);
        h->ms_last = res;
      }
      __atomic_fetch_add(&h->stats[0], (int64_t)res.launches, __ATOMIC_RELAXED);
      if (res.status != 1) {  // 0 finished; 2 failed, info set
        if (scaled) PSD_CUDA(psd::ms::postscale(stream, aux.ms, n, p, Ap, rc.wantT, dEig + (size_t)b * 2 * n));
        continue;
      }
      // no convergence: the iteration drained its bulges, so the factors are still
      // Hessenberg-triangular with Z accumulated; the single-bulge team kernel finishes this problem
    }
    if (batch == 1) {
      team_needed = true;
    } else {
      RealCall r1 = rc;
      if ((e = launch_team_iteration(h, dev, aux, stream, r1, 1, Ab, Zb, dEig + (size_t)b * 2 * n, dInfo + b))) return e;
      if (scaled) PSD_CUDA(psd::ms::postscale(stream, aux.ms, n, p, Ap, rc.wantT, dEig + (size_t)b * 2 * n));
    }
  }
  if (team_needed) {
    if ((e = launch_team_iteration(h, dev, aux, stream, rc, 1, dA, dZ, dEig, dInfo))) return e;
    if (scaled) {
      double* Ap[psd::LH_MAXP];
      for (int j = 1; j <= p; j++) Ap[j - 1] = dA + (size_t)((rc.left ? (p + 1 - j) : j) - 1) * nn;
      PSD_CUDA(psd::ms::postscale(stream, aux.ms, n, p, Ap, rc.wantT, dEig));
    }
  }
  __atomic_fetch_add(&h->stats[2], (int64_t)batch, __ATOMIC_RELAXED);
  return PSD_OK;
}

// On an error inside a shard loop: wait for every slot stream of the device (copies into the
// caller's buffers may still be in flight) before the call returns.
int drain_slots(Device& dev, int code) {
  const std::string keep = g_err;
  for (int k = 0; k < kSlotsPerDevice; k++)
    if (dev.slots[k].stream) cudaStreamSynchronize(dev.slots[k].stream);
  cudaGetLastError();
  g_err = keep;
  return code;
}
#define PSD_SHARD_CUDA(call)                                                                        \
  do {                                                                                              \
    cudaError_t e__ = (call);                                                                       \
    if (e__ != cudaSuccess)                                                                         \
      return drain_slots(dev, fail(PSD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__))); \
  } while (0)

// One host array of a batched call as the pipeline copies it: problem b's part starts at
// host + b * per.
struct HostArray {
  char* host;           // nullptr: a device buffer the kernels write but the call does not return
  size_t per;           // bytes per problem
  Role role;            // the slot buffers it goes through
  bool pinned = true;   // false: staged even when the call runs pinned
  bool counted = true;  // counted in the h2d / d2h bytes
};

// Enqueues the kernels of one chunk of nb problems on the slot's stream; d[role] is the chunk's
// device buffer of each listed array (nullptr for the other roles).
using LaunchFn = std::function<int(Slot& s, long long nb, void* const* d)>;

// One device's share of a batched host call: the problems from `first` on, in `chunks`.  Chunk c
// runs on slot c % kSlotsPerDevice.  A pinned call copies the caller's buffers in place; otherwise
// they go through the slot's pinned staging buffers.  `in` lists the factors first.
int run_shard(Device& dev, long long first, const std::vector<long long>& chunks, bool pinned,
              const std::vector<HostArray>& in, const std::vector<HostArray>& out, const LaunchFn& launch,
              int64_t* bytes_h2d, int64_t* bytes_d2h) {
  // chunks above this size are copied straight from / to pageable memory (no pinned staging copy)
  const size_t kStageLimit = 1ULL << 30;
  // results of a staged chunk that still sit in a slot's pinned buffers: copied out when the slot
  // is drained (before its next use, or at the end), so that the host copies overlap the device
  // work of the other slots
  struct Pending {
    char* dst;
    const void* src;
    size_t bytes;
  };
  std::vector<Pending> pend[kSlotsPerDevice];
  auto flush = [&](int k) {
    for (const Pending& q : pend[k]) std::memcpy(q.dst, q.src, q.bytes);
    pend[k].clear();
  };
  long long off = first;
  for (size_t c = 0; c < chunks.size(); off += chunks[c++]) {
    const long long nb = chunks[c];
    const int si = (int)(c % kSlotsPerDevice);
    Slot& s = dev.slots[si];
    if (!s.stream) PSD_SHARD_CUDA(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    // the slot's previous chunk must have fully drained before its buffers are reused
    PSD_SHARD_CUDA(cudaStreamSynchronize(s.stream));
    flush(si);
    const bool big = nb * in[0].per > kStageLimit;
    auto staged = [&](const HostArray& a) { return pinned ? !a.pinned : !big; };
    int e;
    void* d[kRoles] = {};
    for (const auto* list : {&in, &out})
      for (const HostArray& a : *list) {
        if ((e = ensure_dev(s.dBuf[a.role], s.dCap[a.role], nb * a.per))) return drain_slots(dev, e);
        d[a.role] = s.dBuf[a.role];
      }
    for (const HostArray& a : in) {
      const char* src = a.host + off * a.per;
      const size_t bytes = nb * a.per;
      const bool st = staged(a);
      if (st) {
        if ((e = ensure_pinned(s.hBuf[a.role], s.hCap[a.role], bytes))) return drain_slots(dev, e);
        std::memcpy(s.hBuf[a.role], src, bytes);
      }
      PSD_SHARD_CUDA(cudaMemcpyAsync(d[a.role], st ? s.hBuf[a.role] : src, bytes, cudaMemcpyHostToDevice, s.stream));
      if (a.counted) *bytes_h2d += (int64_t)bytes;
    }
    if ((e = launch(s, nb, d))) return drain_slots(dev, e);
    for (const HostArray& a : out) {
      if (!a.host) continue;
      char* dst = a.host + off * a.per;
      const size_t bytes = nb * a.per;
      const bool st = staged(a);
      if (st && (e = ensure_pinned(s.hBuf[a.role], s.hCap[a.role], bytes))) return drain_slots(dev, e);
      PSD_SHARD_CUDA(cudaMemcpyAsync(st ? s.hBuf[a.role] : dst, d[a.role], bytes, cudaMemcpyDeviceToHost, s.stream));
      if (st) pend[si].push_back({dst, s.hBuf[a.role], bytes});
      if (a.counted) *bytes_d2h += (int64_t)bytes;
    }
  }
  for (int k = 0; k < kSlotsPerDevice; k++)
    if (dev.slots[k].stream) {
      PSD_SHARD_CUDA(cudaStreamSynchronize(dev.slots[k].stream));
      flush(k);
    }
  return PSD_OK;
}

// Runs one device's share [first, first + count) of a batched host call, on the current device.
using ShardFn = std::function<int(Device& dev, long long first, long long count, bool pinned, int64_t* bytes_h2d,
                                  int64_t* bytes_d2h)>;

// A batched host call: one contiguous range of the batch per device of the handle, each on a host
// thread of its own.  The call runs pinned when every buffer in `args` is page-locked.
int run_host(psd_handle_s* h, int64_t batch, std::initializer_list<const void*> args, const ShardFn& shard) {
  std::lock_guard<std::mutex> lock(h->mu);
  for (auto& s : h->stats) s = 0;
  if (batch == 0) return PSD_OK;
  bool pinned = true;
  for (const void* a : args) pinned = pinned && is_pinned(a);
  const int nd = (int)h->devs.size();
  std::vector<int> codes(nd, PSD_OK);
  std::vector<std::string> msgs(nd);
  std::vector<int64_t> h2d(nd, 0), d2h(nd, 0);
  auto t0 = std::chrono::steady_clock::now();
  auto run_device = [&](int d) -> int {
    const long long lo = batch * d / nd, hi = batch * (d + 1) / nd;
    if (hi == lo) return PSD_OK;
    PSD_CUDA(cudaSetDevice(h->devs[d].ordinal));
    return shard(h->devs[d], lo, hi - lo, pinned, &h2d[d], &d2h[d]);
  };
  auto work = [&](int d) {
    if ((codes[d] = run_device(d))) msgs[d] = g_err;
  };
  if (nd == 1) {
    work(0);
  } else {
    std::vector<std::thread> th;
    for (int d = 0; d < nd; d++) th.emplace_back(work, d);
    for (auto& t : th) t.join();
  }
  auto t1 = std::chrono::steady_clock::now();
  for (int d = 0; d < nd; d++) {
    h->stats[3] += h2d[d];
    h->stats[4] += d2h[d];
  }
  h->stats[5] = std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
  for (int d = 0; d < nd; d++)
    if (codes[d]) return fail(codes[d], msgs[d]);
  return PSD_OK;
}

// Chunk sizes of the real standard path for `count` problems of `per` bytes of factors.
// Chunks grow geometrically (x4) from 1/16 of the full size up to ~2 GiB of factors: the first
// host-to-device copy is the only one no kernel overlaps, so it is kept short, while the large
// later chunks amortise the tail of the persistent kernels (measured on config 2).
std::vector<long long> plan_real_chunks(long long count, size_t per, bool pinned) {
  long long chunk = std::max<long long>(1, (2048LL << 20) / (long long)per);
  if (!pinned) chunk = std::max<long long>(1, std::min<long long>(chunk, (512LL << 20) / (long long)per));
  chunk = std::min(chunk, count);
  // pageable buffers are staged through pinned ones by the host: at least four chunks, so that the
  // host copies of one chunk overlap the device work of the others
  if (!pinned && (size_t)count * per >= (64u << 20) && count >= 8)
    chunk = std::min(chunk, (count + 3) / 4);
  std::vector<long long> chunks;
  long long next = (count > chunk) ? std::max<long long>(1, chunk / (pinned ? 16 : 2)) : chunk;
  for (long long off = 0; off < count; off += chunks.back()) {
    chunks.push_back(std::min(next, count - off));
    next = std::min(chunk, next * 4);
  }
  return chunks;
}

int run_real_host(psd_handle_t h, const RealCall& rc, int64_t batch, double* A, double* Z, double* eig,
                  int32_t* info) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  if (rc.n < 1 || rc.p < 1 || batch < 0) return fail(PSD_ERR_BAD_ARG, "n, p must be >= 1 and batch >= 0");
  if (!A) return fail(PSD_ERR_BAD_ARG, "A must not be NULL");
  if (!rc.reduce_only && (!eig || !info)) return fail(PSD_ERR_BAD_ARG, "eig and info must not be NULL");
  if (rc.wantZ && !Z) return fail(PSD_ERR_BAD_ARG, "wantZ set but Z is NULL");
  if (h->devs.empty()) return fail(PSD_ERR_NO_DEVICE, "handle has no CUDA device");
  const size_t per = (size_t)rc.n * rc.n * rc.p * sizeof(double);  // bytes of factors per problem
  const bool wantZ = rc.wantZ && Z;
  return run_host(h, batch, {A, Z, eig, info}, [&](Device& dev, long long first, long long count, bool pinned,
                                                   int64_t* bytes_h2d, int64_t* bytes_d2h) {
    std::vector<HostArray> in{{(char*)A, per, kFactors}}, out;
    if (wantZ && rc.z_preset) in.push_back({(char*)Z, per, kZ});  // Z enters as the caller's Q_j (accumulated onto)
    if (rc.wantT || rc.reduce_only) out.push_back({(char*)A, per, kFactors});
    if (wantZ) out.push_back({(char*)Z, per, kZ});
    if (!rc.reduce_only) {
      out.push_back({(char*)eig, 2 * rc.n * sizeof(double), kVal0});
      out.push_back({(char*)info, sizeof(int32_t), kInfo});
      // the iteration counts are a setting of the handle, not an argument of the call: they do not
      // decide whether the call runs pinned, and the byte counters leave them out
      int32_t* it = h->iters_host;
      if (it) out.push_back({(char*)it, sizeof(int32_t), kIters, is_pinned(it), false});
    }
    auto launch = [&](Slot& s, long long nb, void* const* d) -> int {
      int32_t* iters = (int32_t*)d[kIters];
      if (iters) PSD_CUDA(cudaMemsetAsync(iters, 0, nb * sizeof(int32_t), s.stream));
      s.curIters = iters;
      const int e = launch_real(h, dev, s, s.stream, rc, nb, (double*)d[kFactors], (double*)d[kZ],
                                (double*)d[kVal0], (int32_t*)d[kInfo]);
      s.curIters = nullptr;
      return e;
    };
    return run_shard(dev, first, plan_real_chunks(count, per, pinned), pinned, in, out, launch, bytes_h2d,
                     bytes_d2h);
  });
}


// ---------------------------------------------------------------------------------------------
// Generalized paths (complex periodic QZ; real periodic QZ): the pipeline of the real standard
// path with a chunk policy of their own, and (alpha, beta, alphascale) instead of eig.
// ---------------------------------------------------------------------------------------------
struct GenCall {
  int n, p, left, wantT, wantZ, maxitfac, skip_reduce;
  int cplx;                 // 1: complex128 factors, complex beta; 0: real factors, real beta
  const unsigned char* S;   // host, user order
  int reduce_only = 0;
};

size_t gen_elem(const GenCall& gc) { return gc.cplx ? 16 : 8; }

template <class T>
int launch_gen_t(psd_handle_s* h, Device& dev, Slot& aux, cudaStream_t stream, const GenCall& gc, long long batch,
                 void* dA, void* dZ, void* dAlpha, void* dBeta, long long* dScale, int32_t* dInfo) {
  const int n = gc.n, p = gc.p;
  const bool wantZ = gc.wantZ && dZ;
  int e = ensure_dev(aux.dS, aux.capS, (size_t)p);
  if (e) return e;
  PSD_CUDA(cudaMemcpyAsync(aux.dS, gc.S, (size_t)p, cudaMemcpyHostToDevice, stream));
  if (!aux.dCounter) PSD_CUDA(cudaMalloc((void**)&aux.dCounter, 2 * sizeof(unsigned long long)));
  PSD_CUDA(cudaMemsetAsync(aux.dCounter, 0, sizeof(unsigned long long), stream));
  int optin = 0;
  PSD_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev.ordinal));
  int threads = ((2 * n + 31) / 32) * 32;
  threads = std::max(64, std::min(threads, 256));
  // Two instantiations: 255 registers (one 256-thread CTA per SM) and 128 registers (two).  With the
  // factors in global memory the second resident problem pays: while one CTA walks its rotation
  // chains (one warp busy) the other streams its strips (profiles/r1_gen_variants.txt).
  // (Factors in shared memory: always the 255-register one.)
  auto kern = psd::gpschur_kernel<T, 256>;
  cudaFuncAttributes fa;
  PSD_CUDA(cudaFuncGetAttributes(&fa, kern));
  const size_t max_dyn = (size_t)optin - fa.sharedSizeBytes;
  const size_t small = (size_t)((psd::cq_small_doubles(n, p) + 1) & ~1LL) * sizeof(double);
  const int ldh = (sizeof(T) == 8 && n % 2 == 0) ? n + 1 : n;  // odd leading dimension for real data
  const size_t mats = (size_t)p * ldh * n * sizeof(T) * (wantZ ? 2 : 1);
  psd::GpqzParams<T> P;
  P.n = n; P.p = p; P.batch = batch; P.left = gc.left; P.wantT = gc.wantT; P.wantZ = wantZ ? 1 : 0;
  P.maxitfac = gc.maxitfac > 0 ? gc.maxitfac : (gc.cplx ? 30 : 120);  // generalized.jl:169, rgeneralized.jl:52
  P.skip_reduce = gc.skip_reduce;
  P.reduce_only = gc.reduce_only;
  P.blocked_stage1 = 0;
  P.windowed_stage2 = 0;
  P.windowed_qz = 0;
  P.S = aux.dS;
  P.A = (T*)dA; P.Z = wantZ ? (T*)dZ : nullptr;
  P.alpha = (psd::cplx*)dAlpha; P.beta = (T*)dBeta; P.scale = dScale; P.info = dInfo;
  P.counter = aux.dCounter;
  P.debug = dbg_env("PSD_GEN_PROF") ? 1 : 0;
  size_t smem;
  if (small + mats <= max_dyn) {
    P.use_smem = 1; P.ldh = ldh; smem = small + mats;
    P.deep = dbg_env("PSD_DEEP_SMEM") ? 1 : 0;
  } else {
    if (small > max_dyn) return fail(PSD_ERR_UNSUPPORTED, "n or p too large for the per-CTA state");
    P.use_smem = 0; P.ldh = n; smem = small;
    // table-driven single-pass chases (items in flight per thread), measured as above: a gain for
    // the complex path, a small loss for the real one
    P.deep = (sizeof(T) == sizeof(psd::cplx)) ? 2 : 0;
    if (dbg_env("PSD_NO_DEEP")) P.deep = 0;
    if (const char* ev = dbg_env("PSD_DEEP_U")) P.deep = atoi(ev);
    const size_t blk = (size_t)psd::blk_work_scalars(n) * sizeof(T);
    if (!gc.skip_reduce && small + blk <= max_dyn && !dbg_env("PSD_NO_BLOCKED_STAGE1")) {
      P.blocked_stage1 = 1;
      smem = small + blk;
    }
    const size_t qzw = sizeof(T) == sizeof(double) ? (size_t)psd::qzw_work_doubles(p, psd::S3_K_CTA) * sizeof(double)
                                                   : (size_t)psd::s4_work_scalars<T>(p) * sizeof(T);
    if (!gc.reduce_only && small + qzw <= max_dyn && !dbg_env("PSD_NO_WINDOWED_QZ")) {
      P.windowed_qz = 1;
      smem = std::max(smem, small + qzw);
    }
    const size_t s2w = (size_t)psd::s2_work_scalars(p) * sizeof(T);
    if (!gc.skip_reduce && small + s2w <= max_dyn && !dbg_env("PSD_NO_WINDOWED_STAGE2")) {
      P.windowed_stage2 = 1;
      smem = std::max(smem, small + s2w);
    }
  }
  bool wide = !P.use_smem;
  if (const char* ev = dbg_env("PSD_GEN_WIDE")) wide = atoi(ev) != 0;
  if (const char* ev = dbg_env("PSD_GEN_THREADS")) threads = std::max(64, std::min(atoi(ev), wide ? 512 : 256));
  if (wide) kern = psd::gpschur_kernel<T, 512>;
  PSD_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_dyn));
  int occ = 0;
  PSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem));
  if (occ < 1) return fail(PSD_ERR_UNSUPPORTED, "kernel does not fit on an SM");
  const int grid = (int)std::max(1LL, std::min((long long)occ * dev.sm_count, batch));
  {
    ScopedKernelTimer tm(h, dev, stream, 1);
    kern<<<grid, threads, smem, stream>>>(P);
  }
  PSD_CUDA(cudaGetLastError());
  __atomic_fetch_add(&h->stats[0], (int64_t)1, __ATOMIC_RELAXED);
  __atomic_fetch_add(&h->stats[P.use_smem ? 1 : 2], (int64_t)batch, __ATOMIC_RELAXED);
  return PSD_OK;
}

int launch_gen(psd_handle_s* h, Device& dev, Slot& aux, cudaStream_t stream, const GenCall& gc, long long batch,
               void* dA, void* dZ, void* dAlpha, void* dBeta, long long* dScale, int32_t* dInfo) {
  if (batch == 0) return PSD_OK;
  if (gc.cplx)
    return launch_gen_t<psd::cplx>(h, dev, aux, stream, gc, batch, dA, dZ, dAlpha, dBeta, dScale, dInfo);
  return launch_gen_t<double>(h, dev, aux, stream, gc, batch, dA, dZ, dAlpha, dBeta, dScale, dInfo);
}

// Chunk sizes of the generalized paths for `count` problems of `per` bytes of factors and
// `dev_per` bytes of device buffers.  One CTA works on one problem (for seconds at the larger
// orders), so a launch should carry at least two problems per SM; beyond that, 512 MiB of factors
// per launch keeps the copies of one chunk under the kernels of the others.  The cap keeps the
// slots inside device memory.
int plan_gen_chunks(const Device& dev, long long count, size_t per, size_t dev_per, std::vector<long long>& chunks) {
  long long chunk = std::max<long long>(1, (512LL << 20) / (long long)per);
  const long long wave = 2LL * dev.sm_count;  // resident problems per launch in global-memory mode
  chunk = (chunk + wave - 1) / wave * wave;   // whole waves: no half-empty tail inside a launch
  size_t free_b = 0, total_b = 0;
  PSD_CUDA(cudaMemGetInfo(&free_b, &total_b));
  const long long cap = (long long)((total_b / 2) / kSlotsPerDevice / dev_per);
  chunk = std::min(std::max<long long>(1, std::min(chunk, cap)), count);
  for (long long off = 0; off < count; off += chunk) chunks.push_back(std::min(chunk, count - off));
  return PSD_OK;
}

int run_gen_host(psd_handle_t h, const GenCall& gc, int64_t batch, void* A, void* Z, void* alpha, void* beta,
                 int64_t* scale, int32_t* info) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  if (gc.n < 1 || gc.p < 1 || batch < 0) return fail(PSD_ERR_BAD_ARG, "n, p must be >= 1 and batch >= 0");
  if (!A || !gc.S) return fail(PSD_ERR_BAD_ARG, "A and S must not be NULL");
  if (!gc.reduce_only && (!alpha || !beta || !scale || !info))
    return fail(PSD_ERR_BAD_ARG, "alpha, beta, alphascale and info must not be NULL");
  if (gc.wantZ && !Z) return fail(PSD_ERR_BAD_ARG, "wantZ set but Z is NULL");
  // leftmost factor after orientation must have S = true (generalized.jl:140, rgeneralized.jl:37)
  if (!gc.S[gc.left ? gc.p - 1 : 0]) return fail(PSD_ERR_SIGNATURE, "The leftmost entry in S must be true");
  if (h->devs.empty()) return fail(PSD_ERR_NO_DEVICE, "handle has no CUDA device");
  const size_t es = gen_elem(gc);
  const size_t per = (size_t)gc.n * gc.n * gc.p * es;  // bytes of factors per problem
  const size_t xB[3] = {(size_t)gc.n * 16, (size_t)gc.n * es, (size_t)gc.n * 8};  // alpha, beta, alphascale
  const bool wantZ = gc.wantZ && Z;
  return run_host(h, batch, {A, Z, alpha, beta, scale, info}, [&](Device& dev, long long first, long long count,
                                                                  bool pinned, int64_t* bytes_h2d, int64_t* bytes_d2h) {
    std::vector<long long> chunks;
    if (int e = plan_gen_chunks(dev, count, per, per * (wantZ ? 2 : 1) + (xB[0] + xB[1] + xB[2]) + 64, chunks))
      return e;
    std::vector<HostArray> in{{(char*)A, per, kFactors}}, out;
    if (gc.wantT) out.push_back({(char*)A, per, kFactors});
    if (wantZ) out.push_back({(char*)Z, per, kZ});
    if (!gc.reduce_only) {
      out.push_back({(char*)alpha, xB[0], kVal0});
      out.push_back({(char*)beta, xB[1], kVal1});
      out.push_back({(char*)scale, xB[2], kVal2});
    }
    // the reduction-only kernel writes info as well, which the call does not return
    out.push_back({gc.reduce_only ? nullptr : (char*)info, sizeof(int32_t), kInfo});
    auto launch = [&](Slot& s, long long nb, void* const* d) {
      return launch_gen(h, dev, s, s.stream, gc, nb, d[kFactors], d[kZ], d[kVal0], d[kVal1], (long long*)d[kVal2],
                        (int32_t*)d[kInfo]);
    };
    return run_shard(dev, first, chunks, pinned, in, out, launch, bytes_h2d, bytes_d2h);
  });
}

}  // namespace

extern "C" {

int psd_version(void) { return PSD_VERSION; }

int psd_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

const char* psd_last_error_string(void) { return g_err.c_str(); }

int psd_create(psd_handle_t* handle, int ndev, const int* devices) {
  if (!handle) return fail(PSD_ERR_BAD_ARG, "handle pointer is NULL");
  *handle = nullptr;
  int avail = psd_device_count();
  if (avail <= 0) return fail(PSD_ERR_NO_DEVICE, "no CUDA device visible (this library has no CPU fallback)");
  std::vector<int> ords;
  if (ndev <= 0) {
    for (int i = 0; i < avail; i++) ords.push_back(i);
  } else {
    if (!devices) return fail(PSD_ERR_BAD_ARG, "devices is NULL");
    for (int i = 0; i < ndev; i++) {
      if (devices[i] < 0 || devices[i] >= avail) return fail(PSD_ERR_BAD_ARG, "device ordinal out of range");
      ords.push_back(devices[i]);
    }
  }
  auto* h = new (std::nothrow) psd_handle_s;
  if (!h) return fail(PSD_ERR_BAD_ARG, "out of host memory");
  for (int o : ords) {
    Device d;
    d.ordinal = o;
    cudaDeviceProp prop;
    cudaError_t e = cudaGetDeviceProperties(&prop, o);
    if (e != cudaSuccess) {
      delete h;
      return fail(PSD_ERR_CUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
    }
    if (prop.major < 10) {
      delete h;
      return fail(PSD_ERR_NO_DEVICE, "device is not sm_100 class (this library is built for sm_100a only)");
    }
    d.sm_count = prop.multiProcessorCount;
    h->devs.push_back(d);
  }
  *handle = h;
  return PSD_OK;
}

int psd_destroy(psd_handle_t h) {
  if (!h) return PSD_OK;
  for (auto& d : h->devs) {
    cudaSetDevice(d.ordinal);
    auto freeSlot = [](Slot& s) {
      if (s.stream) {
        cudaStreamSynchronize(s.stream);
        cudaStreamDestroy(s.stream);
      }
      for (int k = 0; k < kRoles; k++) {
        cudaFree(s.dBuf[k]);
        cudaFreeHost(s.hBuf[k]);
      }
      cudaFree(s.dCounter); cudaFree(s.dScratch); cudaFree(s.dPacked); cudaFree(s.dS);
      for (int k = 0; k < 8; k++) cudaFree(s.dPk[k]);
      cudaFree(s.dPhaseCtr);
      cudaFree(s.dProf);
      psd::ms::ws_destroy(s.ms);
      for (int k = 0; k < 3; k++) {
        cudaFree(s.dArg[k]);
        cudaFree(s.dTeam[k]);
      }
    };
    for (auto& s : d.slots) freeSlot(s);
    freeSlot(d.user);
    if (d.userDone) cudaEventDestroy(d.userDone);
  }
  cudaGetLastError();
  delete h;
  return PSD_OK;
}

int psd_handle_device_count(psd_handle_t h) { return h ? (int)h->devs.size() : 0; }

int psd_rpschur_batched(psd_handle_t h, int n, int p, int64_t batch, int orientation, int wantT,
                        int wantZ, int maxitfac, double* A, double* Z, double* eig, int32_t* info) {
  if (orientation != 0 && orientation != 1)
    return fail(PSD_ERR_BAD_ARG, "orientation argument must be either 0 (:R, right) or 1 (:L, left)");
  RealCall rc{n, p, orientation, wantT != 0, wantZ != 0, maxitfac, 0, 0};
  return run_real_host(h, rc, batch, A, Z, eig, info);
}

int psd_rpschur_hessut_batched(psd_handle_t h, int n, int p, int64_t batch, int wantT, int wantZ,
                               int maxitfac, double* A, double* Z, double* eig, int32_t* info) {
  RealCall rc{n, p, 0, wantT != 0, wantZ != 0, maxitfac, 0, 1};
  return run_real_host(h, rc, batch, A, Z, eig, info);
}

int psd_rpschur_hessut_q_batched(psd_handle_t h, int n, int p, int64_t batch, int wantT, int maxitfac, double* A,
                                 double* Q, double* eig, int32_t* info) {
  if (!Q) return fail(PSD_ERR_BAD_ARG, "Q must not be NULL");
  RealCall rc{n, p, 0, wantT != 0, 1, maxitfac, 0, 1};
  rc.z_preset = 1;
  return run_real_host(h, rc, batch, A, Q, eig, info);
}

int psd_rcheckpsd_batched(psd_handle_t h, int n, int p, int64_t batch, int orientation, const double* A,
                          const double* T, const double* Z, double* err, double* tri, double* orth) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  if (n < 1 || p < 1 || batch < 0 || !A || !T || !Z || !err) return fail(PSD_ERR_BAD_ARG, "bad argument");
  if (orientation != 0 && orientation != 1) return fail(PSD_ERR_BAD_ARG, "bad orientation");
  if (h->devs.empty()) return fail(PSD_ERR_NO_DEVICE, "handle has no CUDA device");
  std::lock_guard<std::mutex> lock(h->mu);
  if (batch == 0) return PSD_OK;
  if (int e = use_slot0(h)) return e;
  Device& dev = h->devs[0];
  Slot& s = dev.slots[0];
  const size_t per = (size_t)n * n * p;
  // a diagnostic, not a hot path: plain chunks of at most ~1 GiB per array, synchronous copies
  const long long chunk = std::max<long long>(1, std::min<long long>(batch, (1LL << 30) / (long long)(per * sizeof(double))));
  double *dA = nullptr, *dT = nullptr, *dZ = nullptr, *dOut = nullptr;
  std::vector<double> hout((size_t)chunk * p * 4);
  auto cleanup = [&] { cudaFree(dA); cudaFree(dT); cudaFree(dZ); cudaFree(dOut); };
#define PSD_CHK(call)                                                    \
  do {                                                                   \
    cudaError_t e__ = (call);                                            \
    if (e__ != cudaSuccess) {                                            \
      cleanup();                                                         \
      return fail(PSD_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); \
    }                                                                    \
  } while (0)
  PSD_CHK(cudaMalloc((void**)&dA, chunk * per * sizeof(double)));
  PSD_CHK(cudaMalloc((void**)&dT, chunk * per * sizeof(double)));
  PSD_CHK(cudaMalloc((void**)&dZ, chunk * per * sizeof(double)));
  PSD_CHK(cudaMalloc((void**)&dOut, chunk * p * 4 * sizeof(double)));
  const int CB = (n <= 1024) ? 4 : 1;
  const size_t smem = (size_t)2 * n * CB * sizeof(double);
  if (CB == 4)
    PSD_CHK(cudaFuncSetAttribute(psd::checkpsd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  else
    PSD_CHK(cudaFuncSetAttribute(psd::checkpsd_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const double eps = 2.220446049250313e-16;
  for (long long off = 0; off < batch; off += chunk) {
    const long long nb = std::min(chunk, batch - off);
    PSD_CHK(cudaMemcpyAsync(dA, A + (size_t)off * per, nb * per * sizeof(double), cudaMemcpyHostToDevice, s.stream));
    PSD_CHK(cudaMemcpyAsync(dT, T + (size_t)off * per, nb * per * sizeof(double), cudaMemcpyHostToDevice, s.stream));
    PSD_CHK(cudaMemcpyAsync(dZ, Z + (size_t)off * per, nb * per * sizeof(double), cudaMemcpyHostToDevice, s.stream));
    PSD_CHK(cudaMemsetAsync(dOut, 0, nb * p * 4 * sizeof(double), s.stream));
    psd::CheckParams P;
    P.n = n; P.p = p; P.left = orientation; P.batch = nb;
    P.A = dA; P.T = dT; P.Z = dZ; P.out = dOut;
    // enough CTAs to fill the device a few times over
    long long zc = std::max<long long>(1, std::min<long long>((n + CB - 1) / CB, (4LL * dev.sm_count + nb * p - 1) / (nb * p)));
    P.cols_per_cta = (int)(((n + zc - 1) / zc + CB - 1) / CB * CB);
    zc = (n + P.cols_per_cta - 1) / P.cols_per_cta;
    for (long long b0 = 0; b0 < nb; b0 += 32768) {  // grid.y limit
      const long long by = std::min<long long>(32768, nb - b0);
      psd::CheckParams Q = P;
      Q.A = dA + (size_t)b0 * per; Q.T = dT + (size_t)b0 * per; Q.Z = dZ + (size_t)b0 * per;
      Q.out = dOut + (size_t)b0 * p * 4;
      if (CB == 4)
        psd::checkpsd_kernel<4><<<dim3(p, (unsigned)by, (unsigned)zc), 256, smem, s.stream>>>(Q);
      else
        psd::checkpsd_kernel<1><<<dim3(p, (unsigned)by, (unsigned)zc), 256, smem, s.stream>>>(Q);
    }
    PSD_CHK(cudaGetLastError());
    PSD_CHK(cudaMemcpyAsync(hout.data(), dOut, nb * p * 4 * sizeof(double), cudaMemcpyDeviceToHost, s.stream));
    PSD_CHK(cudaStreamSynchronize(s.stream));
    for (long long k = 0; k < nb * p; k++) {
      const double e2 = hout[4 * k], a1 = hout[4 * k + 1], t2 = hout[4 * k + 2], o2 = hout[4 * k + 3];
      err[off * p + k] = (a1 > 0.0) ? std::sqrt(e2) / eps / a1 : (e2 > 0.0 ? HUGE_VAL : 0.0);
      if (tri) tri[off * p + k] = std::sqrt(t2);
      if (orth) orth[off * p + k] = std::sqrt(o2);
    }
  }
#undef PSD_CHK
  cleanup();
  return PSD_OK;
}

int psd_rphess_packed_batched(psd_handle_t h, int n, int p, int64_t batch, double* A, double* tau) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  if (n < 1 || p < 1 || batch < 0 || !A || !tau) return fail(PSD_ERR_BAD_ARG, "bad argument");
  if (h->devs.empty()) return fail(PSD_ERR_NO_DEVICE, "handle has no CUDA device");
  std::lock_guard<std::mutex> lock(h->mu);
  if (batch == 0) return PSD_OK;
  if (int e = use_slot0(h)) return e;
  Device& dev = h->devs[0];
  Slot& s = dev.slots[0];
  const size_t per = (size_t)n * n * p;
  const long long chunk = std::max<long long>(1, std::min<long long>(batch, (1LL << 30) / (long long)(per * sizeof(double))));
  int e;
  if ((e = ensure_dev(s.dArg[0], s.capArg[0], chunk * per * sizeof(double)))) return e;
  if ((e = ensure_dev(s.dArg[1], s.capArg[1], std::max<size_t>((size_t)chunk * p * n, (size_t)chunk * 2 * n) * sizeof(double)))) return e;
  if ((e = ensure_dev(s.dArg[2], s.capArg[2], chunk * sizeof(int32_t)))) return e;
  RealCall rc{n, p, 0, 1, 0, 30, 1, 0};
  for (long long off = 0; off < batch; off += chunk) {
    const long long nb = std::min(chunk, batch - off);
    PSD_CUDA(cudaMemcpyAsync(s.dArg[0], A + (size_t)off * per, nb * per * sizeof(double), cudaMemcpyHostToDevice, s.stream));
    s.curTau = s.dArg[1];
    e = launch_real(h, dev, s, s.stream, rc, nb, s.dArg[0], nullptr, nullptr, (int32_t*)s.dArg[2]);
    s.curTau = nullptr;
    if (e) return e;
    PSD_CUDA(cudaMemcpyAsync(A + (size_t)off * per, s.dArg[0], nb * per * sizeof(double), cudaMemcpyDeviceToHost, s.stream));
    PSD_CUDA(cudaMemcpyAsync(tau + (size_t)off * p * n, s.dArg[1], nb * p * n * sizeof(double), cudaMemcpyDeviceToHost, s.stream));
    PSD_CUDA(cudaStreamSynchronize(s.stream));
  }
  return PSD_OK;
}

int psd_host_alloc(size_t bytes, int write_combined, void** out) {
  if (!out || bytes == 0) return fail(PSD_ERR_BAD_ARG, "bad argument");
  *out = nullptr;
  const unsigned flags = cudaHostAllocPortable | (write_combined ? cudaHostAllocWriteCombined : 0u);
  cudaError_t e = cudaHostAlloc(out, bytes, flags);
  if (e != cudaSuccess) return fail(PSD_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e));
  return PSD_OK;
}

int psd_host_free(void* ptr) {
  if (!ptr) return PSD_OK;
  cudaError_t e = cudaFreeHost(ptr);
  if (e != cudaSuccess) return fail(PSD_ERR_CUDA, std::string("cudaFreeHost: ") + cudaGetErrorString(e));
  return PSD_OK;
}

int psd_set_iters_output(psd_handle_t h, int32_t* iters) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  std::lock_guard<std::mutex> lock(h->mu);
  h->iters_host = iters;
  return PSD_OK;
}

int psd_rphess_batched(psd_handle_t h, int n, int p, int64_t batch, int wantQ, double* A, double* Q) {
  RealCall rc{n, p, 0, 1, wantQ != 0, 30, 1, 0};
  return run_real_host(h, rc, batch, A, Q, nullptr, nullptr);
}

int psd_rpschur_batched_dev(psd_handle_t h, int dev_index, void* stream, int n, int p, int64_t batch,
                            int orientation, int wantT, int wantZ, int maxitfac, double* dA,
                            double* dZ, double* deig, int32_t* dinfo) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  if (dev_index < 0 || dev_index >= (int)h->devs.size()) return fail(PSD_ERR_BAD_ARG, "dev_index out of range");
  if (n < 1 || p < 1 || batch < 0 || !dA || !deig || !dinfo) return fail(PSD_ERR_BAD_ARG, "bad argument");
  if (orientation != 0 && orientation != 1) return fail(PSD_ERR_BAD_ARG, "bad orientation");
  if (wantZ && !dZ) return fail(PSD_ERR_BAD_ARG, "wantZ set but dZ is NULL");
  std::lock_guard<std::mutex> lock(h->mu);
  Device& dev = h->devs[dev_index];
  PSD_CUDA(cudaSetDevice(dev.ordinal));
  cudaStream_t st = (cudaStream_t)stream;
  if (!st) {
    if (!dev.user.stream) PSD_CUDA(cudaStreamCreateWithFlags(&dev.user.stream, cudaStreamNonBlocking));
    st = dev.user.stream;
  }
  // Every *_dev call on this device uses the same scratch set (work counters, packed buffers):
  // a call waits for the previous one, whatever stream that was enqueued on.
  if (!dev.userDone) PSD_CUDA(cudaEventCreateWithFlags(&dev.userDone, cudaEventDisableTiming));
  else PSD_CUDA(cudaStreamWaitEvent(st, dev.userDone, 0));
  RealCall rc{n, p, orientation, wantT != 0, wantZ != 0, maxitfac, 0, 0};
  const int rcode = launch_real(h, dev, dev.user, st, rc, batch, dA, dZ, deig, dinfo);
  PSD_CUDA(cudaEventRecord(dev.userDone, st));
  return rcode;
}

int psd_cpschur_batched(psd_handle_t h, int n, int p, int64_t batch, int orientation, const uint8_t* S, int wantT,
                        int wantZ, int maxitfac, double* A, double* Z, double* alpha, double* beta,
                        int64_t* alphascale, int32_t* info) {
  if (orientation != 0 && orientation != 1)
    return fail(PSD_ERR_BAD_ARG, "orientation argument must be either 0 (:R, right) or 1 (:L, left)");
  GenCall gc{n, p, orientation, wantT != 0, wantZ != 0, maxitfac, 0, 1, S};
  return run_gen_host(h, gc, batch, A, Z, alpha, beta, alphascale, info);
}

int psd_cpschur_hessut_batched(psd_handle_t h, int n, int p, int64_t batch, const uint8_t* S, int wantT, int wantZ,
                               int maxitfac, double* A, double* Z, double* alpha, double* beta,
                               int64_t* alphascale, int32_t* info) {
  GenCall gc{n, p, 0, wantT != 0, wantZ != 0, maxitfac, 1, 1, S};
  return run_gen_host(h, gc, batch, A, Z, alpha, beta, alphascale, info);
}

int psd_gphess_batched(psd_handle_t h, int cplx, int n, int p, int64_t batch, const uint8_t* S, int wantQ, double* A,
                       double* Q) {
  GenCall gc{n, p, 0, 1, wantQ != 0, 0, 0, cplx != 0, S};
  gc.reduce_only = 1;
  return run_gen_host(h, gc, batch, A, Q, nullptr, nullptr, nullptr, nullptr);
}

int psd_rgpschur_batched(psd_handle_t h, int n, int p, int64_t batch, int orientation, const uint8_t* S, int wantT,
                         int wantZ, int maxitfac, double* A, double* Z, double* alpha, double* beta,
                         int64_t* alphascale, int32_t* info) {
  if (orientation != 0 && orientation != 1)
    return fail(PSD_ERR_BAD_ARG, "orientation argument must be either 0 (:R, right) or 1 (:L, left)");
  GenCall gc{n, p, orientation, wantT != 0, wantZ != 0, maxitfac, 0, 0, S};
  return run_gen_host(h, gc, batch, A, Z, alpha, beta, alphascale, info);
}

int psd_rgpschur_hessut_batched(psd_handle_t h, int n, int p, int64_t batch, const uint8_t* S, int wantT,
                                int wantZ, int maxitfac, double* A, double* Z, double* alpha, double* beta,
                                int64_t* alphascale, int32_t* info) {
  GenCall gc{n, p, 0, wantT != 0, wantZ != 0, maxitfac, 1, 0, S};
  return run_gen_host(h, gc, batch, A, Z, alpha, beta, alphascale, info);
}

int psd_rphess_rowwise_batched(psd_handle_t h, int n, int extra_row, int p, int qrows, int64_t batch, double* Ap,
                               double* A, double* Q) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  if (n < 1 || p < 1 || batch < 0 || !Ap || (p > 1 && !A) || (Q && qrows < 1))
    return fail(PSD_ERR_BAD_ARG, "bad argument");
  if (h->devs.empty()) return fail(PSD_ERR_NO_DEVICE, "handle has no CUDA device");
  std::lock_guard<std::mutex> lock(h->mu);
  for (auto& s : h->stats) s = 0;
  if (batch == 0) return PSD_OK;
  if (int e = use_slot0(h)) return e;
  Device& dev = h->devs[0];
  Slot& s = dev.slots[0];
  const int m = n + (extra_row ? 1 : 0);
  const size_t bAp = (size_t)batch * m * n * sizeof(double);
  const size_t bA = (size_t)batch * (p - 1) * n * n * sizeof(double);
  const size_t bQ = Q ? (size_t)batch * p * qrows * n * sizeof(double) : 0;
  int e;
  if ((e = ensure_dev(s.dArg[0], s.capArg[0], bAp))) return e;
  if (bA && (e = ensure_dev(s.dArg[1], s.capArg[1], bA))) return e;
  if (bQ && (e = ensure_dev(s.dArg[2], s.capArg[2], bQ))) return e;
  PSD_CUDA(cudaMemcpyAsync(s.dArg[0], Ap, bAp, cudaMemcpyHostToDevice, s.stream));
  if (bA) PSD_CUDA(cudaMemcpyAsync(s.dArg[1], A, bA, cudaMemcpyHostToDevice, s.stream));
  if (bQ) PSD_CUDA(cudaMemcpyAsync(s.dArg[2], Q, bQ, cudaMemcpyHostToDevice, s.stream));
  psd::RowHessParams<double> P;
  P.n = n; P.m = m; P.p = p; P.qrows = qrows; P.batch = batch;
  P.Ap = s.dArg[0]; P.A = bA ? s.dArg[1] : nullptr; P.Q = bQ ? s.dArg[2] : nullptr;
  const int threads = std::max(64, std::min(256, ((std::max(n, qrows) + 31) / 32) * 32));
  const int grid = (int)std::min<long long>(batch, (long long)dev.sm_count * 4);
  {
    ScopedKernelTimer tm(h, dev, s.stream, 0);
    psd::rowhess_kernel<double><<<grid, threads, (size_t)(n + 2) * sizeof(double), s.stream>>>(P);
  }
  PSD_CUDA(cudaGetLastError());
  PSD_CUDA(cudaMemcpyAsync(Ap, s.dArg[0], bAp, cudaMemcpyDeviceToHost, s.stream));
  if (bA) PSD_CUDA(cudaMemcpyAsync(A, s.dArg[1], bA, cudaMemcpyDeviceToHost, s.stream));
  if (bQ) PSD_CUDA(cudaMemcpyAsync(Q, s.dArg[2], bQ, cudaMemcpyDeviceToHost, s.stream));
  PSD_CUDA(cudaStreamSynchronize(s.stream));
  h->stats[0] = 1;
  h->stats[2] = batch;
  h->stats[3] = (int64_t)(bAp + bA + bQ);
  h->stats[4] = (int64_t)(bAp + bA + bQ);
  return PSD_OK;
}

int psd_dgemm_host(psd_handle_t h, int transA, int transB, int M, int N, int K, double alpha, const double* A,
                   int lda, const double* B, int ldb, double beta, double* C, int ldc, int reps, double* ms) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  if (M < 0 || N < 0 || K < 0 || !A || !B || !C) return fail(PSD_ERR_BAD_ARG, "bad argument");
  if (h->devs.empty()) return fail(PSD_ERR_NO_DEVICE, "handle has no CUDA device");
  std::lock_guard<std::mutex> lock(h->mu);
  if (int e = use_slot0(h)) return e;
  Device& dev = h->devs[0];
  Slot& s = dev.slots[0];
  const size_t bA = (size_t)lda * (transA ? M : K) * 8, bB = (size_t)ldb * (transB ? K : N) * 8;
  const size_t bC = (size_t)ldc * N * 8;
  int e;
  if ((e = ensure_dev(s.dArg[0], s.capArg[0], bA))) return e;
  if ((e = ensure_dev(s.dArg[1], s.capArg[1], bB))) return e;
  if ((e = ensure_dev(s.dArg[2], s.capArg[2], bC))) return e;
  PSD_CUDA(cudaMemcpyAsync(s.dArg[0], A, bA, cudaMemcpyHostToDevice, s.stream));
  PSD_CUDA(cudaMemcpyAsync(s.dArg[1], B, bB, cudaMemcpyHostToDevice, s.stream));
  PSD_CUDA(cudaMemcpyAsync(s.dArg[2], C, bC, cudaMemcpyHostToDevice, s.stream));
  psd::GemmArgs g;
  g.M = M; g.N = N; g.K = K;
  g.A = s.dArg[0]; g.rsA = transA ? lda : 1; g.csA = transA ? 1 : lda;
  g.B = s.dArg[1]; g.rsB = transB ? ldb : 1; g.csB = transB ? 1 : ldb;
  g.C = s.dArg[2]; g.ldc = ldc; g.alpha = alpha; g.beta = beta; g.splitK = 1;
  PSD_CUDA(psd::dgemm_launch(s.stream, dev.sm_count, g));
  PSD_CUDA(cudaMemcpyAsync(C, s.dArg[2], bC, cudaMemcpyDeviceToHost, s.stream));
  PSD_CUDA(cudaStreamSynchronize(s.stream));
  if (reps > 0 && ms) {
    cudaEvent_t e0, e1;
    PSD_CUDA(cudaEventCreate(&e0));
    PSD_CUDA(cudaEventCreate(&e1));
    for (int w = 0; w < 3; w++) PSD_CUDA(psd::dgemm_launch(s.stream, dev.sm_count, g));
    PSD_CUDA(cudaEventRecord(e0, s.stream));
    for (int r = 0; r < reps; r++) PSD_CUDA(psd::dgemm_launch(s.stream, dev.sm_count, g));
    PSD_CUDA(cudaEventRecord(e1, s.stream));
    PSD_CUDA(cudaEventSynchronize(e1));
    float f = 0.f;
    PSD_CUDA(cudaEventElapsedTime(&f, e0, e1));
    *ms = f / reps;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
  }
  return PSD_OK;
}

__global__ void fill_uniform_kernel(uint64_t seed, int n, int p, long long batch, long long first_b,
                                    int cplx, double* A) {
  const long long nn = (long long)n * n;
  const long long total = batch * p * nn;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const long long b = e / (p * nn);
    const long long rem = e - b * p * nn;
    const int j = (int)(rem / nn);
    const int c = (int)((rem % nn) / n), r = (int)(rem % n);
    if (cplx) {
      A[2 * e] = psd::gen_uniform(seed, (uint64_t)(first_b + b), j, r, c, 0);
      A[2 * e + 1] = psd::gen_uniform(seed, (uint64_t)(first_b + b), j, r, c, 1);
    } else {
      A[e] = psd::gen_uniform(seed, (uint64_t)(first_b + b), j, r, c, 0);
    }
  }
}

int psd_fill_uniform_host(uint64_t seed, int n, int p, int64_t batch, int64_t first_b, int cplx,
                          double* A) {
  if (n < 1 || p < 1 || batch < 0 || !A) return fail(PSD_ERR_BAD_ARG, "bad argument");
  const long long nn = (long long)n * n;
  unsigned hw = std::thread::hardware_concurrency();
  int nth = (int)std::max(1u, std::min(hw ? hw : 1u, 64u));
  if (batch < nth) nth = (int)std::max<int64_t>(1, batch);
  auto work = [&](int t) {
    const long long lo = batch * t / nth, hi = batch * (t + 1) / nth;
    for (long long b = lo; b < hi; b++)
      for (int j = 0; j < p; j++)
        for (int c = 0; c < n; c++)
          for (int r = 0; r < n; r++) {
            const long long e = (b * p + j) * nn + (long long)c * n + r;
            if (cplx) {
              A[2 * e] = psd::gen_uniform(seed, (uint64_t)(first_b + b), j, r, c, 0);
              A[2 * e + 1] = psd::gen_uniform(seed, (uint64_t)(first_b + b), j, r, c, 1);
            } else {
              A[e] = psd::gen_uniform(seed, (uint64_t)(first_b + b), j, r, c, 0);
            }
          }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nth; t++) th.emplace_back(work, t);
  work(0);
  for (auto& t : th) t.join();
  return PSD_OK;
}

int psd_fill_uniform_dev(void* stream, uint64_t seed, int n, int p, int64_t batch, int64_t first_b,
                         int cplx, double* dA) {
  if (n < 1 || p < 1 || batch < 0 || !dA) return fail(PSD_ERR_BAD_ARG, "bad argument");
  if (batch == 0) return PSD_OK;
  fill_uniform_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(seed, n, p, batch, first_b, cplx, dA);
  PSD_CUDA(cudaGetLastError());
  return PSD_OK;
}

int psd_set_profiling(psd_handle_t h, int on) {
  if (!h) return fail(PSD_ERR_BAD_ARG, "null handle");
  std::lock_guard<std::mutex> lock(h->mu);
  h->profiling = on != 0;
  return PSD_OK;
}

int psd_kernel_times(psd_handle_t h, double ms[8]) {
  if (!h || !ms) return fail(PSD_ERR_BAD_ARG, "null argument");
  std::lock_guard<std::mutex> lock(h->mu);
  std::lock_guard<std::mutex> lk(h->tmu);
  for (int i = 0; i < 8; i++) ms[i] = 0.0;
  ms[6] = h->gemm_flops;
  h->gemm_flops = 0.0;
  ms[7] = h->extra_launches;
  h->extra_launches = 0.0;
  for (auto& t : h->timers) {
    cudaSetDevice(t.ordinal);
    cudaError_t e = cudaEventSynchronize(t.e1);
    float f = 0.f;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&f, t.e0, t.e1);
    cudaEventDestroy(t.e0);
    cudaEventDestroy(t.e1);
    if (e != cudaSuccess) {
      h->timers.clear();
      return fail(PSD_ERR_CUDA, std::string("kernel timer: ") + cudaGetErrorString(e));
    }
    if (t.kind < 2) {
      ms[t.kind] += f;
      ms[2 + t.kind] += 1.0;
    } else {
      ms[2 + t.kind] += f;  // ms[4] = panel kernels, ms[5] = GEMM groups
    }
  }
  h->timers.clear();
  return PSD_OK;
}

int psd_large_stats(psd_handle_t h, double out[16]) {
  if (!h || !out) return fail(PSD_ERR_BAD_ARG, "null argument");
  std::lock_guard<std::mutex> lk(h->tmu);
  const psd::ms::Result& r = h->ms_last;
  for (int i = 0; i < 16; i++) out[i] = 0.0;
  out[0] = r.status; out[1] = r.sweeps; out[2] = (double)r.rounds; out[3] = (double)r.windows;
  out[4] = (double)r.shift_pairs; out[5] = r.exceptional; out[6] = r.final_blocks; out[7] = (double)r.launches;
  out[8] = r.apply_flops; out[9] = r.ms_chase; out[10] = r.ms_apply; out[11] = r.ms_shifts; out[12] = r.ms_scan;
  out[13] = r.ms_final;
  out[14] = r.ms_rounds;
  out[15] = r.host_seconds;
  return PSD_OK;
}

int psd_last_stats(psd_handle_t h, int64_t stats[8]) {
  if (!h || !stats) return fail(PSD_ERR_BAD_ARG, "null argument");
  std::lock_guard<std::mutex> lock(h->mu);
  for (int i = 0; i < 8; i++) stats[i] = h->stats[i];
  return PSD_OK;
}

}  // extern "C"
