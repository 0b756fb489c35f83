// Host interface of the large-N multishift periodic QR iteration (psd_ms.cu), used by the C ABI
// translation unit (psd_capi.cu).  Internal to the library.
#pragma once
#include <cuda_runtime.h>

#include <cstdlib>
#include <string>

namespace psd {
namespace ms {

// Experiment switches (PSD_MS_* environment variables) exist only in builds made with
// -DPSD_DEBUG_ENV; the product library never reads the environment.
inline const char* dbg_env(const char* name) {
#ifdef PSD_DEBUG_ENV
  return getenv(name);
#else
  (void)name;
  return nullptr;
#endif
}

constexpr int kMaxPeriod = 12;  // = MS_MAXP of psd_ms_core.cuh

struct Workspace;  // device + pinned buffers, grown on demand, owned by a handle slot
Workspace* ws_create();
void ws_destroy(Workspace* ws);

struct Result {
  int status = 0;        // 0 finished, 1 no convergence (valid Hessenberg-triangular state left),
                         // 2 failed (*dInfo = n; the state is not usable for a fallback)
  int sweeps = 0;
  long long rounds = 0, windows = 0, shift_pairs = 0;
  int exceptional = 0, final_blocks = 0;
  long long launches = 0;
  double apply_flops = 0.0;  // flops of the tensor-core window updates
  // device milliseconds by kind (only with profile != 0): chase, apply, shifts, scan, final
  double ms_chase = 0.0, ms_apply = 0.0, ms_shifts = 0.0, ms_scan = 0.0, ms_final = 0.0;
  double host_seconds = 0.0;  // wall time of the pipeline (host clock, excludes the collection of profile events)
  double ms_rounds = 0.0;  // sum over the rounds of (first kernel start .. scan kernel end)
};

// largest period / smallest order this path takes
bool supported(int n, int p);

// Power-of-two normalisation of the p factors before the reduction and its inverse afterwards
// (T factors and eigenvalues), see ms_maxabs_kernel.
cudaError_t prescale(cudaStream_t st, Workspace* ws, int n, int p, double* const* A);
cudaError_t postscale(cudaStream_t st, Workspace* ws, int n, int p, double* const* A, int wantT, double* dEig);

// Periodic QR iteration on Hessenberg-triangular factors H[0..p-1] (internal rightwards order,
// column-major, ld = n), Z[j] preset to the Q_j of the reduction (or nullptr).  Eigenvalues to
// dEig[n][2]; *dInfo gets max(*dInfo, failing level).  maxitfac (<= 0: 30) scales the cap on the
// rounds of the iteration.  Synchronises the stream internally.
cudaError_t iterate(cudaStream_t st, int sm_count, Workspace* ws, int n, int p, double* const* H,
                    double* const* Z, int wantT, int wantZ, int maxitfac, double* dEig, int* dInfo,
                    int profile, Result* res);

}  // namespace ms
}  // namespace psd
