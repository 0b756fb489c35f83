// CUDA backend + host entry of the large-N multishift periodic QR iteration.
// Algorithm: psd_ms_core.cuh (bulge chase in diagonal windows), psd_ms_driver.hpp (sweep loop),
// psd_ms_kernels.cuh (kernels).  Compiled as its own translation unit and linked into
// libpsd_b200.so; called from launch_real_large in psd_capi.cu.
#include "psd_ms.h"

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include "psd_ms_driver.hpp"
#include "psd_ms_kernels.cuh"

namespace psd {
namespace ms {

constexpr int kPlanRing = 8;     // rounds whose window lists may be in flight (> lag + 1)
constexpr int kScanRing = 16;    // scan results in flight
constexpr int kShiftSlots = 8;   // shift sets in flight (one side stream each)
constexpr int kMaxWin = MS_MAXCHAINS;

struct Workspace {
  double* dU = nullptr;  size_t capU = 0;        // [2][p][n * W]: accumulated window transformations, by round parity
  double* dPairs = nullptr;                      // [kShiftSlots][66][4] shift pairs
  double* dSnap = nullptr; size_t capSnap = 0;   // [kShiftSlots][p * 64 * 64] trailing-block snapshots
  WinDesc* dPlan = nullptr;                      // [kPlanRing][kMaxWin]
  WinDesc* dList = nullptr; size_t capList = 0;  // final block list
  int* dCtl = nullptr;                           // [kScanRing][8] scan results, [.. + kShiftSlots] pair counts, misc
  double* dSc = nullptr;                         // [2 * MS_MAXP] scales
  unsigned long long* dMax = nullptr;            // [MS_MAXP]
  int* hCtl = nullptr;                           // pinned mirror of dCtl
  // Mapped pinned host memory, read / written by the kernels directly (no copy-engine operation
  // between the kernels of a round): window lists of the rounds in flight, scan results.
  WinDesc* hPlan = nullptr;                      // [kPlanRing][kMaxWin]
  int* hScan = nullptr;                          // [kScanRing][8]: ilo, ihi, done, nzero
  cudaEvent_t evScan[kScanRing] = {nullptr};     // scan kernel done (main stream)
  cudaEvent_t evPub[kScanRing] = {nullptr};      // its result has reached the host (publish stream)
  cudaStream_t pub = nullptr;                    // carries the device -> host copies of the scan results
  cudaStream_t main = nullptr;                   // the pipeline's own stream: highest priority, so that its
                                                 // kernels are never queued behind the shift computations
  cudaEvent_t evIn = nullptr, evOut = nullptr;   // ordering against the caller's stream
  cudaEvent_t evSnap[kShiftSlots] = {nullptr}, evShift[kShiftSlots] = {nullptr};
  cudaStream_t side[kShiftSlots] = {nullptr};
  long long scan_counter = 0;                    // scans issued so far (all calls)
  cudaStream_t scan = nullptr;                   // stand-alone deflation scans (split rounds), high priority
  cudaStream_t far = nullptr;                    // far window updates of a round, concurrent with the next chase
  cudaEvent_t evNear[2] = {nullptr, nullptr}, evFar[2] = {nullptr, nullptr}, evChase[2] = {nullptr, nullptr};
};
constexpr int kScanInts = MS_SCAN_INTS;            // ints per scan result
static_assert(kShiftSlots == MS_SHIFT_SLOTS, "shift slot count");
constexpr int kCtlInts = kScanRing * kScanInts + MS_SS_INTS + 16;
constexpr int kCtlPairs = kScanRing * kScanInts;   // shift supply state (MS_SS_* offsets)
constexpr int kCtlMisc = kScanRing * kScanInts + MS_SS_INTS;  // [0] expo of the scaling, [1] number of final blocks

Workspace* ws_create() { return new Workspace(); }

void ws_destroy(Workspace* ws) {
  if (!ws) return;
  cudaFree(ws->dU); cudaFree(ws->dPairs); cudaFree(ws->dSnap); cudaFree(ws->dPlan); cudaFree(ws->dList);
  cudaFree(ws->dCtl); cudaFree(ws->dSc); cudaFree(ws->dMax);
  cudaFreeHost(ws->hCtl); cudaFreeHost(ws->hPlan); cudaFreeHost(ws->hScan);
  for (auto& e : ws->evScan) if (e) cudaEventDestroy(e);
  for (auto& e : ws->evPub) if (e) cudaEventDestroy(e);
  if (ws->pub) cudaStreamDestroy(ws->pub);
  if (ws->main) cudaStreamDestroy(ws->main);
  if (ws->far) cudaStreamDestroy(ws->far);
  if (ws->scan) cudaStreamDestroy(ws->scan);
  for (int k = 0; k < 2; k++) {
    if (ws->evNear[k]) cudaEventDestroy(ws->evNear[k]);
    if (ws->evFar[k]) cudaEventDestroy(ws->evFar[k]);
    if (ws->evChase[k]) cudaEventDestroy(ws->evChase[k]);
  }
  if (ws->evIn) cudaEventDestroy(ws->evIn);
  if (ws->evOut) cudaEventDestroy(ws->evOut);
  for (int k = 0; k < kShiftSlots; k++) {
    if (ws->evSnap[k]) cudaEventDestroy(ws->evSnap[k]);
    if (ws->evShift[k]) cudaEventDestroy(ws->evShift[k]);
    if (ws->side[k]) cudaStreamDestroy(ws->side[k]);
  }
  delete ws;
}

static_assert(kMaxPeriod == MS_MAXP, "psd_ms.h and psd_ms_core.cuh disagree");

bool supported(int n, int p) { return p >= 1 && p <= MS_MAXP && n >= 2 * geom_for(p).W; }

namespace {

#define MS_CHECK(call)                      \
  do {                                      \
    cudaError_t e__ = (call);               \
    if (e__ != cudaSuccess) return e__;     \
  } while (0)

template <class T>
cudaError_t grow(T*& ptr, size_t& cap, size_t bytes) {
  if (bytes <= cap) return cudaSuccess;
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cap = 0;
  cudaError_t e = cudaMalloc((void**)&ptr, bytes);
  if (e == cudaSuccess) cap = bytes;
  return e;
}

cudaError_t ws_basic(Workspace* ws) {
  if (!ws->dCtl) MS_CHECK(cudaMalloc((void**)&ws->dCtl, kCtlInts * sizeof(int)));
  if (!ws->dSc) MS_CHECK(cudaMalloc((void**)&ws->dSc, 2 * MS_MAXP * sizeof(double)));
  if (!ws->dMax) MS_CHECK(cudaMalloc((void**)&ws->dMax, MS_MAXP * sizeof(unsigned long long)));
  if (!ws->hCtl) MS_CHECK(cudaHostAlloc((void**)&ws->hCtl, kCtlInts * sizeof(int), cudaHostAllocDefault));
  if (!ws->dPairs) MS_CHECK(cudaMalloc((void**)&ws->dPairs, (size_t)kShiftSlots * 66 * 4 * sizeof(double)));
  if (!ws->dPlan) MS_CHECK(cudaMalloc((void**)&ws->dPlan, (size_t)kPlanRing * kMaxWin * sizeof(WinDesc)));
  if (!ws->hPlan)
    MS_CHECK(cudaHostAlloc((void**)&ws->hPlan, (size_t)kPlanRing * kMaxWin * sizeof(WinDesc), cudaHostAllocMapped | cudaHostAllocPortable));
  if (!ws->hScan) MS_CHECK(cudaHostAlloc((void**)&ws->hScan, (size_t)kScanRing * kScanInts * sizeof(int), cudaHostAllocDefault));
  for (auto& e : ws->evScan) if (!e) MS_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  for (auto& e : ws->evPub) if (!e) MS_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  if (!ws->pub) MS_CHECK(cudaStreamCreateWithFlags(&ws->pub, cudaStreamNonBlocking));
  if (!ws->main) {
    int lo = 0, hi = 0;  // lo = least, hi = greatest priority (numerically smaller)
    MS_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    MS_CHECK(cudaStreamCreateWithPriority(&ws->main, cudaStreamNonBlocking, hi));
  }
  if (!ws->scan) {
    int lo = 0, hi = 0;
    MS_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    MS_CHECK(cudaStreamCreateWithPriority(&ws->scan, cudaStreamNonBlocking, hi));
  }
  if (!ws->far) MS_CHECK(cudaStreamCreateWithFlags(&ws->far, cudaStreamNonBlocking));
  for (int k = 0; k < 2; k++) {
    if (!ws->evNear[k]) MS_CHECK(cudaEventCreateWithFlags(&ws->evNear[k], cudaEventDisableTiming));
    if (!ws->evFar[k]) MS_CHECK(cudaEventCreateWithFlags(&ws->evFar[k], cudaEventDisableTiming));
    if (!ws->evChase[k]) MS_CHECK(cudaEventCreateWithFlags(&ws->evChase[k], cudaEventDisableTiming));
  }
  if (!ws->evIn) MS_CHECK(cudaEventCreateWithFlags(&ws->evIn, cudaEventDisableTiming));
  if (!ws->evOut) MS_CHECK(cudaEventCreateWithFlags(&ws->evOut, cudaEventDisableTiming));
  for (int k = 0; k < kShiftSlots; k++) {
    if (!ws->evSnap[k]) MS_CHECK(cudaEventCreateWithFlags(&ws->evSnap[k], cudaEventDisableTiming));
    if (!ws->evShift[k]) MS_CHECK(cudaEventCreateWithFlags(&ws->evShift[k], cudaEventDisableTiming));
    if (!ws->side[k]) MS_CHECK(cudaStreamCreateWithFlags(&ws->side[k], cudaStreamNonBlocking));
  }
  return cudaSuccess;
}

struct Timer {  // optional per-launch timing (profile mode only)
  bool on = false;
  cudaStream_t st;
  std::vector<cudaEvent_t> ev;
  std::vector<int> kind;
  int begin(int k) {
    if (!on) return -1;
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, st);
    ev.push_back(a);
    ev.push_back(b);
    kind.push_back(k);
    return (int)kind.size() - 1;
  }
  void end(int id = -2) {
    if (!on) return;
    if (id == -2) id = (int)kind.size() - 1;
    if (id >= 0) cudaEventRecord(ev[2 * id + 1], st);
  }
  // gaps[a * 6 + b]: device time between the end of a kernel of kind a and the start of the next
  // timed kernel (kind b) on the stream
  void collect_gaps(double* gaps) {
    int prev = -1;
    for (size_t i = 0; i < kind.size(); i++) {
      if (kind[i] == 5) continue;
      if (prev >= 0) {
        float f = 0.f;
        cudaEventSynchronize(ev[2 * i]);
        if (cudaEventElapsedTime(&f, ev[2 * prev + 1], ev[2 * i]) == cudaSuccess) gaps[kind[prev] * 6 + kind[i]] += f;
      }
      prev = (int)i;
    }
  }
  void collect(double* ms) {
    for (size_t i = 0; i < kind.size(); i++) {
      float f = 0.f;
      cudaEventSynchronize(ev[2 * i + 1]);
      cudaEventElapsedTime(&f, ev[2 * i], ev[2 * i + 1]);
      ms[kind[i]] += f;
      cudaEventDestroy(ev[2 * i]);
      cudaEventDestroy(ev[2 * i + 1]);
    }
    ev.clear();
    kind.clear();
  }
};

struct CudaBackend {
  cudaStream_t st;
  int sm_count;
  Workspace* ws;
  int n, p, wantT, wantZ, maxitfac;
  Geom g;
  double* H[MS_MAXP];
  double* Z[MS_MAXP];
  double* dEig;
  int* dInfo;
  size_t chase_smem, shift_smem, block_smem;
  cudaError_t err = cudaSuccess;
  long long launches = 0;
  long long nscan = 0, nplan = 0;
  int scan_seq[kScanRing] = {0};
  long long* dProf = nullptr;
  int round_timer = -1;
  bool slot_used[kShiftSlots] = {false};
  Timer tm, tm_far, tm_side[kShiftSlots];
  long long nround = 0;
  // debug: device timeline of a few rounds (PSD_MS_TIMELINE=<first round>)
  long long tl_first = -1;
  int tl_cnt = 0;
  std::vector<cudaEvent_t> tl_ev;
  std::vector<std::string> tl_name;
  void mark(const char* name, cudaStream_t s) {
    if (tl_first == -1) return;
    if (tl_first >= 0 && (nround < tl_first || nround >= tl_first + 4)) return;
    if (tl_first < -1 && (nround % 64) >= 2) return;  // sampling mode: two consecutive rounds out of 64
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, s);
    tl_ev.push_back(e);
    tl_name.push_back(std::string(name) + " r" + std::to_string(nround) + " w" + std::to_string(tl_cnt));
  }
  void timeline_print() {
    for (size_t i = 0; i < tl_ev.size(); i++) {
      float f = 0.f;
      cudaEventSynchronize(tl_ev[i]);
      cudaEventElapsedTime(&f, tl_ev[0], tl_ev[i]);
      fprintf(stderr, "[psd ms timeline] %8.1f us  %s\n", f * 1e3, tl_name[i].c_str());
      }
    for (auto e : tl_ev) cudaEventDestroy(e);
    tl_ev.clear();
  }
  bool split = true;  // far updates on their own stream
  bool scan_used = false;
  cudaEvent_t pending_scan_ev = nullptr;
  double wait_scan = 0.0, wait_shift = 0.0, wait_plan = 0.0;  // host seconds blocked on the device
  struct Stopwatch {
    double& acc;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    explicit Stopwatch(double& a) : acc(a) {}
    ~Stopwatch() { acc += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); }
  };

  bool ok() const { return err == cudaSuccess; }
  void note(cudaError_t e) {
    if (err == cudaSuccess && e != cudaSuccess) err = e;
  }
  int shift_slots() const { return kShiftSlots; }
  bool trace() const { return dbg_env("PSD_MS_TRACE") != nullptr; }
  int max_windows() const { return kMaxWin; }
  int pair_offset(int slot) const { return slot * 66; }

  // Scan of the subdiagonal after a round (wins = that round's windows, already on the device in
  // the plan slot used last); the result lands in a pinned ring slot.
  const WinDesc* last_plan = nullptr;
  // The scan kernel leaves its result and then its sequence number in device memory.  The host
  // polls for it with small copies on a side stream that has NO dependency on the main stream: an
  // event (or a write to mapped host memory) after the scan kernel was measured to delay the next
  // kernel of the main stream by 100 - 140 us (device clock), i.e. a quarter of a round.
  int fused_slot = -1;  // scan already enqueued as the tail of the round's last update kernel
  int next_scan_slot() {
    const int slot = (int)(nscan % kScanRing);
    nscan++;
    // sequence numbers are unique over the life of the workspace: the result slots keep the values
    // of earlier calls, and a repeated number would make the host take a stale result for the new one
    scan_seq[slot] = (int)(++ws->scan_counter & 0x3fffffff) + 1;
    return slot;
  }
  int scan_async(const WinDesc* /*host copy, unused here*/, int cnt, int nmin) {
    if (fused_slot >= 0) {
      const int slot = fused_slot;
      fused_slot = -1;
      if (round_timer >= 0) tm.end(round_timer);
      round_timer = -1;
      return slot;
    }
    const int slot = next_scan_slot();
    if (!ok()) return slot;
    tm.begin(3);
    ms_scan_kernel<<<1, 1024, (size_t)2 * n + 16, st>>>(H[0], n, nmin, ws->dCtl + slot * kScanInts, scan_seq[slot], last_plan,
                                                          last_plan ? cnt : 0, g.W, g.D, dProf);
    tm.end();
    if (round_timer >= 0) tm.end(round_timer);
    round_timer = -1;
    launches++;
    note(cudaGetLastError());
    return slot;
  }
  void scan_wait(int slot, ScanInfo& info) {
    if (!ok()) { info.done = 1; return; }
    {
      Stopwatch sw(wait_scan);
      int* h = ws->hScan + slot * kScanInts;
      bool seen = false;
      for (long long spins = 0;; spins++) {
        note(cudaMemcpyAsync(h, ws->dCtl + slot * kScanInts, kScanInts * sizeof(int), cudaMemcpyDeviceToHost, ws->pub));
        note(cudaStreamSynchronize(ws->pub));
        if (!ok()) break;
        if (seen) break;                 // second copy after the sequence number: every field is final
        if (h[4] == scan_seq[slot]) { seen = true; continue; }
        if ((spins & 0xff) == 0xff) {    // a failed launch must not hang the caller
          cudaError_t q = cudaStreamQuery(st);
          if (q == cudaSuccess && scan_used) q = cudaStreamQuery(ws->scan);
          if (q == cudaSuccess) {
            note(cudaMemcpyAsync(h, ws->dCtl + slot * kScanInts, kScanInts * sizeof(int), cudaMemcpyDeviceToHost, ws->pub));
            note(cudaStreamSynchronize(ws->pub));
            if (h[4] != scan_seq[slot]) note(cudaErrorUnknown);
            break;
          }
          if (q != cudaErrorNotReady) { note(q); break; }
        }
      }
    }
    if (!ok()) { info.done = 1; return; }
    const int* c = ws->hScan + slot * kScanInts;
    info.ilo = c[0]; info.ihi = c[1]; info.done = c[2]; info.nzero = c[3];
    info.nb = std::min(c[5], (int)MS_MAXBLK);
    for (int b = 0; b < info.nb; b++) { info.blo[b] = c[6 + 2 * b]; info.bhi[b] = c[7 + 2 * b]; }
  }

  // Shift set: snapshot of the trailing block on the main stream, eigenvalues on a side stream;
  // the kernel publishes the set as "newest" when it is complete.  fence: the main stream waits.
  int shift_seq = 0;
  void shifts_request(int slot, int lo, int m, double perturb, bool fence) {
    if (!ok()) return;
    // the slot's previous computation must have finished before its snapshot is overwritten
    if (slot_used[slot]) note(cudaStreamWaitEvent(st, ws->evShift[slot], 0));
    slot_used[slot] = true;
    double* snap = ws->dSnap + (size_t)slot * p * 64 * 64;
    SnapParams S;
    S.n = n; S.p = p; S.lo = lo; S.m = m; S.snap = snap;
    S.seq_word = ws->dCtl + kCtlPairs + MS_SS_SEQ + slot;
    for (int j = 0; j < p; j++) S.H[j] = H[j];
    ms_snapshot_kernel<<<std::min(64, (p * m * m + 255) / 256), 256, 0, st>>>(S);
    note(cudaGetLastError());
    note(cudaEventRecord(ws->evSnap[slot], st));
    cudaStream_t ss = ws->side[slot];
    note(cudaStreamWaitEvent(ss, ws->evSnap[slot], 0));
    ShiftParams P;
    P.p = p; P.m = m; P.snap = snap;
    P.pairs = ws->dPairs + (size_t)pair_offset(slot) * 4;
    P.state = ws->dCtl + kCtlPairs;
    P.slot = slot; P.seq = ++shift_seq; P.lo = lo;
    P.perturb = perturb;
    tm_side[slot].begin(2);
    ms_shifts_kernel<<<1, 256, shift_smem, ss>>>(P);
    tm_side[slot].end();
    launches += 2;
    note(cudaGetLastError());
    note(cudaEventRecord(ws->evShift[slot], ss));
    if (fence) note(cudaStreamWaitEvent(st, ws->evShift[slot], 0));
  }

  // Window updates of one list of windows.  part 0: everything, on the main stream.  part 1: the
  // tiles next to the windows (main stream, the scan rides on its last CTA).  part 2: the rest, on
  // the far stream.
  // phases: bit 0 = row updates and Z, bit 1 = column updates
  void apply(const WinDesc* wins, int cnt, const double* U, int part, int scan_slot = -1, int phases = 3) {
    cudaStream_t s = (part == 2) ? ws->far : st;
    Timer& t = (part == 2) ? tm_far : tm;
    ApplyParams A;
    A.n = n; A.p = p; A.W = g.W; A.wantT = wantT; A.wantZ = wantZ; A.nwin = cnt;
    A.do_scan = 0; A.scan_nmin = g.W; A.scan_seq = 0; A.scan_D = g.D; A.scan_ctl = nullptr;
    A.scan_ticket = (unsigned int*)(ws->dCtl + kCtlMisc + 4); A.prof = dProf;
    for (int j = 0; j < p; j++) { A.H[j] = H[j]; A.Z[j] = Z[j]; }
    A.U = U; A.wins = wins; A.part = part;
    const int tiles = (n + AP_T - 1) / AP_T;
    // consecutive tiles per CTA (U_j staged once): as many as still leave a few waves of CTAs
    // (about half of the tile slots of an item are empty: left of / below the window)
    int tpb = 1;
    while (tpb < 4 && (long long)(tiles / (2 * tpb)) * cnt * p * 2 >= 6LL * sm_count) tpb *= 2;  // (8: measured slower)
    if (const char* e = dbg_env("PSD_MS_TPB")) { if (atoi(e) > 0) tpb = atoi(e); }
    if (part == 1) tpb = 1;
    A.tpb = tpb;
    // near part: two tiles right of the window, one above it
    const int chunks0 = (part == 1) ? 2 : (tiles + tpb - 1) / tpb;
    const int chunks1 = (part == 1) ? 1 : (tiles + tpb - 1) / tpb;
    t.begin(1);
    if (phases & 1) {
      A.phase = 0;
      ms_apply_kernel<<<dim3(chunks0, cnt * p * 2), 256, AP_SMEM, s>>>(A);
      launches++;
      if (part == 1) mark("near0 end", s);
    }
    if (phases & 2) {
      A.phase = 1;
      if (scan_slot >= 0) {
        A.do_scan = 1;
        A.scan_seq = scan_seq[scan_slot];
        A.scan_ctl = ws->dCtl + scan_slot * kScanInts;
      }
      ms_apply_kernel<<<dim3(chunks1, cnt * p), 256, AP_SMEM, s>>>(A);
      launches++;
    }
    t.end();
    note(cudaGetLastError());
  }

  void round(const std::vector<WinDesc>& wins) {
    if (!ok()) return;
    const int cnt = (int)std::min<size_t>(wins.size(), kMaxWin);
    // The host runs at most `lag` (< kPlanRing - 1) rounds ahead of the scans it has seen, and a
    // scan is enqueued behind the chase kernel that read the slot, so the slot is free again.
    const int slot = (int)(nplan % kPlanRing);
    nplan++;
    WinDesc* hp = ws->hPlan + (size_t)slot * kMaxWin;
    WinDesc* dp = ws->dPlan + (size_t)slot * kMaxWin;
    std::copy(wins.begin(), wins.begin() + cnt, hp);
    __sync_synchronize();
    WinDesc* hp_dev = nullptr;
    note(cudaHostGetDevicePointer((void**)&hp_dev, hp, 0));
    if (!ok()) return;
    ChaseParams C;
    C.n = n; C.p = p; C.g = g;
    for (int j = 0; j < p; j++) C.H[j] = H[j];
    double* Ucur = ws->dU + (size_t)(nround & 1) * p * n * g.W;
    C.U = Ucur; C.shifts = ws->dPairs; C.shift_state = ws->dCtl + kCtlPairs; C.wins = hp_dev; C.wins_dev = dp; C.prof = dProf;
    C.idle_count = ws->dCtl + kCtlMisc + 6;
    if (dProf && dbg_env("PSD_MS_STAMP")) {
      const int mode = atoi(dbg_env("PSD_MS_STAMP"));
      if (mode == 1) ms_stamp_kernel<<<1, 32, 0, st>>>(dProf, 8);
      if (mode == 2) ms_stamp_kernel<<<cnt, 512, chase_smem, st>>>(dProf, 8);
    }
    if (pending_scan_ev) {
      note(cudaStreamWaitEvent(st, pending_scan_ev, 0));
      pending_scan_ev = nullptr;
    }
    round_timer = tm.begin(5);
    tl_cnt = cnt;
    mark("chase begin", st);
    tm.begin(0);
    ms_chase_kernel<<<cnt, 64 * g.NB, chase_smem, st>>>(C);
    tm.end();
    launches++;
    note(cudaGetLastError());
    fused_slot = next_scan_slot();
    // Round r, main stream: chase(r), near0(r), near1(r); far stream: far0(r), far1(r).  near = the
    // two tiles (128 columns) right of a window for its row update (near0) and the tile (64 rows)
    // above it for its column update (near1); far0 / far1 = the other tiles, and all of Z in far0.
    //   far0(r) waits for chase(r) (and, by stream order, far(r-1));  far1(r) also for near(r);
    //   near0(r) waits for far(r-1);  chase(r+1) follows near1(r) and runs beside far(r).
    //  * chase(r+1) cannot touch what far(r) works on: a far entry (i, k) of the row update of a
    //    window [s, s+wl) has k >= s + wl + 128 > i + 128, a far entry of its column update has
    //    i < s - 64 <= k - 64, and a diagonal block of order <= 64 holds no entry with k - i >= 64,
    //    wherever it lies.  The same holds for the shift snapshot (order nsw <= W) and the scan.
    //  * near1(b) and far0(a) never share an entry: rows of a lie in [s_b - 64, s_b) only if
    //    s_b < s_a + wl_a + 64, and then the columns of b end before s_a + wl_a + 128.
    //  * a block rows(a) x cols(b) of two windows a above b gets U_a' from the left and U_b from the
    //    right; piecewise application is correct as long as a left update of a column finds all
    //    rows of a in one state with respect to U_b, and vice versa.  By the previous point the
    //    columns of b are all inside near0(a) when near1(b) reaches rows of a (near0 precedes near1),
    //    and no row of a has seen U_b when far0(a) reaches columns of b.  far1 runs after every left
    //    update of the round.
    //  * near0(r+1) overlaps far(r) (the windows have moved): hence its wait.
    //  * U is double-buffered by round parity: chase(r+2) runs after near(r+1), i.e. after far(r).
    const int par = (int)(nround & 1);
    mark("chase end", st);
    if (split) {
      note(cudaEventRecord(ws->evChase[par], st));
      // the scan reads three diagonals of H_1, which only the chase writes
      note(cudaStreamWaitEvent(ws->scan, ws->evChase[par], 0));
      ms_scan_kernel<<<1, 1024, (size_t)2 * n + 16, ws->scan>>>(H[0], n, g.W, ws->dCtl + fused_slot * kScanInts, scan_seq[fused_slot], dp,
                                                                 cnt, g.W, g.D, dProf);
      launches++;
      note(cudaGetLastError());
      // it also writes the zeros of the deflations: the next chase must see them
      note(cudaEventRecord(ws->evScan[fused_slot], ws->scan));
      pending_scan_ev = ws->evScan[fused_slot];
      scan_used = true;
      note(cudaStreamWaitEvent(ws->far, ws->evChase[par], 0));
      mark("far0 begin", ws->far);
      apply(dp, cnt, Ucur, 2, -1, 1);
      mark("far0 end", ws->far);
      if (nround > 0) note(cudaStreamWaitEvent(st, ws->evFar[par ^ 1], 0));
      mark("near begin", st);
      apply(dp, cnt, Ucur, 1);
      mark("near end", st);
      note(cudaEventRecord(ws->evNear[par], st));
      note(cudaStreamWaitEvent(ws->far, ws->evNear[par], 0));
      apply(dp, cnt, Ucur, 2, -1, 2);
      mark("far1 end", ws->far);
      note(cudaEventRecord(ws->evFar[par], ws->far));
    } else {
      apply(dp, cnt, Ucur, 0, fused_slot);
    }
    nround++;
    last_plan = dp;
  }

  // the far stream joins the main stream
  void join() {
    if (pending_scan_ev) {
      note(cudaStreamWaitEvent(st, pending_scan_ev, 0));
      pending_scan_ev = nullptr;
    }
    if (nround > 0 && split) note(cudaStreamWaitEvent(st, ws->evFar[(nround - 1) & 1], 0));
  }

  void finish(int& nblocks) {
    nblocks = 0;
    join();
    if (!ok()) return;
    note(grow(ws->dList, ws->capList, (size_t)(n / 2 + 1) * sizeof(WinDesc)));
    if (!ok()) return;
    BlockParams B;
    B.n = n; B.p = p; B.W = g.W; B.wantT = wantT; B.wantZ = wantZ; B.maxitfac = maxitfac;
    for (int j = 0; j < p; j++) B.H[j] = H[j];
    B.U = ws->dU; B.eig = dEig; B.info = dInfo; B.list = ws->dList; B.ctl = ws->dCtl + kCtlMisc - 4;
    tm.begin(4);
    ms_blocklist_kernel<<<1, 1024, 0, st>>>(B);
    launches++;
    note(cudaGetLastError());
    note(cudaMemcpyAsync(ws->hCtl + kCtlMisc + 1, ws->dCtl + kCtlMisc + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    note(cudaStreamSynchronize(st));
    if (!ok()) return;
    nblocks = ws->hCtl[kCtlMisc + 1];
    if (nblocks > 0) {
      ms_blocks_kernel<<<std::min(nblocks, sm_count), 256, block_smem, st>>>(B, nblocks);
      launches++;
      note(cudaGetLastError());
    }
    tm.end();
    if (nblocks > 0 && (wantT || wantZ)) {
      // grid.y is limited to 65535: apply in slices of blocks
      const int per = std::max(1, 60000 / (2 * p));
      for (int o = 0; o < nblocks; o += per) apply(ws->dList + o, std::min(per, nblocks - o), ws->dU, 0);
    }
  }
};

}  // namespace

cudaError_t prescale(cudaStream_t st, Workspace* ws, int n, int p, double* const* A) {
  if (p > MS_MAXP) return cudaSuccess;
  MS_CHECK(ws_basic(ws));
  MS_CHECK(cudaMemsetAsync(ws->dMax, 0, MS_MAXP * sizeof(unsigned long long), st));
  const long long cnt = (long long)n * n;
  for (int j = 0; j < p; j++) ms_maxabs_kernel<<<296, 256, 0, st>>>(A[j], cnt, ws->dMax + j);
  ms_scales_kernel<<<1, 32, 0, st>>>(ws->dMax, p, ws->dSc, ws->dCtl + kCtlMisc);
  for (int j = 0; j < p; j++) ms_scale_kernel<<<592, 256, 0, st>>>(A[j], cnt, ws->dSc + j);
  return cudaGetLastError();
}

cudaError_t postscale(cudaStream_t st, Workspace* ws, int n, int p, double* const* A, int wantT, double* dEig) {
  if (p > MS_MAXP) return cudaSuccess;
  const long long cnt = (long long)n * n;
  if (wantT)
    for (int j = 0; j < p; j++) ms_scale_kernel<<<592, 256, 0, st>>>(A[j], cnt, ws->dSc + p + j);
  if (dEig) ms_scale_eig_kernel<<<32, 256, 0, st>>>(dEig, n, ws->dCtl + kCtlMisc);
  return cudaGetLastError();
}

cudaError_t iterate(cudaStream_t caller, int sm_count, Workspace* ws, int n, int p, double* const* H,
                    double* const* Z, int wantT, int wantZ, int maxitfac, double* dEig, int* dInfo,
                    int profile, Result* res) {
  MS_CHECK(ws_basic(ws));
  // the pipeline runs on its own high-priority stream, ordered after / before the caller's stream
  cudaStream_t st = dbg_env("PSD_MS_NO_PRIO") ? caller : ws->main;
  if (st != caller) {
    MS_CHECK(cudaEventRecord(ws->evIn, caller));
    MS_CHECK(cudaStreamWaitEvent(st, ws->evIn, 0));
  }
  CudaBackend be;
  be.st = st; be.sm_count = sm_count; be.ws = ws;
  be.n = n; be.p = p; be.wantT = wantT; be.wantZ = (wantZ && Z) ? 1 : 0;
  be.maxitfac = maxitfac > 0 ? maxitfac : 30;
  be.g = geom_for(p);
  for (int j = 0; j < p; j++) {
    be.H[j] = H[j];
    be.Z[j] = be.wantZ ? Z[j] : nullptr;
  }
  be.dEig = dEig; be.dInfo = dInfo;
  be.tm.on = profile != 0;
  be.tm.st = st;
  be.tm_far.on = profile != 0;
  be.tm_far.st = ws->far;
  if (dbg_env("PSD_MS_NO_SPLIT")) be.split = false;
  if (const char* ev = dbg_env("PSD_MS_TIMELINE")) be.tl_first = atoll(ev);
  const Geom g = be.g;
  MS_CHECK(grow(ws->dU, ws->capU, (size_t)2 * p * n * g.W * sizeof(double)));
  DriverConfig cfg;
  cfg.n = n; cfg.p = p; cfg.wantT = wantT; cfg.wantZ = be.wantZ; cfg.maxitfac = be.maxitfac;
  // Shift window: 12 x 12 (six shift pairs per set).  Larger windows give better Ritz values, but
  // the one-CTA computation takes longer (64 x 64: 14 ms, during which the first launch of every
  // round on the main stream was measured to start 100 - 140 us late), and with dozens of packets
  // in flight every set is stale by many rounds when it is used: measured on three shapes, the
  // shift pairs per eigenvalue and the run time FALL from 48 over 24 to 12 (N = 4096, p = 4:
  // iteration 0.86 / 0.65 / 0.59 s; profiles/r2_large_n_tuning.md).
  int nsw = 12;
  while (nsw > 8 && ((size_t)((rp_small_doubles(nsw, p) + 1) & ~1LL) + (size_t)p * (nsw + 1) * nsw) * 8 > 200 * 1024) nsw -= 4;
  cfg.nsw = nsw;
  if (const char* ev = dbg_env("PSD_MS_REP")) cfg.rep_max = std::max(1, atoi(ev));
  if (const char* ev = dbg_env("PSD_MS_AHEAD")) cfg.sets_ahead = std::max(1, atoi(ev));
  if (const char* ev = dbg_env("PSD_MS_SCAN_EVERY")) cfg.scan_every = std::max(1, atoi(ev));
  if (const char* ev = dbg_env("PSD_MS_MAXBLOCKS")) cfg.max_blocks = std::max(1, atoi(ev));
  if (const char* ev = dbg_env("PSD_MS_NEWDELAY")) cfg.new_block_delay = std::max(0, atoi(ev));
  if (const char* ev = dbg_env("PSD_MS_LAG")) cfg.lag = std::max(1, std::min(kPlanRing - 2, atoi(ev)));
  if (const char* ev = dbg_env("PSD_MS_NSW")) {
    // (the snapshot buffers hold 64 x 64; the far-stream argument needs nsw <= W)
    int want = std::max(2, std::min(std::min(64, g.W), atoi(ev)));
    while (want > 16 && ((size_t)((rp_small_doubles(want, p) + 1) & ~1LL) + (size_t)p * (want + 1) * want) * 8 > 200 * 1024) want -= 8;
    cfg.nsw = want;
  }
  MS_CHECK(grow(ws->dSnap, ws->capSnap, (size_t)kShiftSlots * p * 64 * 64 * sizeof(double)));
  for (int k = 0; k < kShiftSlots; k++) { be.tm_side[k].on = profile != 0; be.tm_side[k].st = ws->side[k]; }
  be.chase_smem = ((size_t)2 * p * g.W * g.LD + (size_t)MS_MAXNB * MS_MAXP * MB_STRIDE) * sizeof(double);
  be.shift_smem = ((size_t)((rp_small_doubles(cfg.nsw, p) + 1) & ~1LL) + (size_t)p * (cfg.nsw + 1) * cfg.nsw) * 8;
  be.block_smem = ((size_t)((rp_small_doubles(g.W, p) + 1) & ~1LL) + (size_t)2 * p * (g.W + 1) * g.W) * 8;
  MS_CHECK(cudaFuncSetAttribute(ms_chase_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)be.chase_smem));
  MS_CHECK(cudaFuncSetAttribute(ms_shifts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)be.shift_smem));
  MS_CHECK(cudaFuncSetAttribute(ms_blocks_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)be.block_smem));
  MS_CHECK(cudaFuncSetAttribute(ms_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AP_SMEM));
  MS_CHECK(cudaFuncSetAttribute(ms_stamp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)be.chase_smem));
  // every kernel of a round asks for the same (largest) shared-memory carve-out, so that the SMs
  // are not reconfigured between the kernels of the pipeline
  if (dbg_env("PSD_MS_SCAN_CARVEOUT")) {
    MS_CHECK(cudaFuncSetAttribute(ms_scan_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    MS_CHECK(cudaFuncSetAttribute(ms_snapshot_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  }
  if (!dbg_env("PSD_MS_NO_CARVEOUT")) {

    MS_CHECK(cudaFuncSetAttribute(ms_apply_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    MS_CHECK(cudaFuncSetAttribute(ms_chase_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
    MS_CHECK(cudaFuncSetAttribute(ms_shifts_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared));
  }
  MS_CHECK(cudaMemsetAsync(ws->dCtl + kCtlPairs, 0, MS_SS_INTS * sizeof(int), st));
  MS_CHECK(cudaMemsetAsync(ws->dCtl + kCtlMisc + 4, 0, 3 * sizeof(int), st));  // scan ticket, -, idle windows
  long long* dprof = nullptr;
  if (dbg_env("PSD_MS_CHASE_PROF")) {
    cudaMalloc((void**)&dprof, 16 * sizeof(long long));
    cudaMemsetAsync(dprof, 0, 16 * sizeof(long long), st);
    be.dProf = dprof;
  }
  DriverStats ds;
  const auto t_drive0 = std::chrono::steady_clock::now();
  const int status = drive(be, cfg, ds);
  be.join();  // (finish() has joined already unless the drive stopped early)
  if (be.tl_first != -1) be.timeline_print();
  const double t_drive = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_drive0).count();
  // side streams: nothing of this call may still be running when the caller reuses the buffers
  for (int k = 0; k < kShiftSlots; k++)
    if (be.slot_used[k]) cudaStreamSynchronize(ws->side[k]);
  cudaStreamSynchronize(ws->pub);
  if (be.scan_used) cudaStreamSynchronize(ws->scan);
  if (st != caller) {
    cudaEventRecord(ws->evOut, st);
    cudaStreamWaitEvent(caller, ws->evOut, 0);
  }
  if (!be.ok()) return be.err;
  if (status == 2) {
    // the drain did not end: the factors may hold bulges, so no fallback may run on them
    const int level = n;
    MS_CHECK(cudaMemcpyAsync(dInfo, &level, sizeof(int), cudaMemcpyHostToDevice, st));
    MS_CHECK(cudaStreamSynchronize(st));
  }
  // windows whose packet had no bulge left (identity U_j): their updates were skipped
  int idle_windows = 0;
  cudaMemcpyAsync(&idle_windows, ws->dCtl + kCtlMisc + 6, sizeof(int), cudaMemcpyDeviceToHost, st);
  cudaStreamSynchronize(st);
  if (ds.windows > 0) ds.apply_flops *= 1.0 - (double)idle_windows / (double)ds.windows;
  if (res) {
    res->status = status;
    res->sweeps = ds.sweeps; res->rounds = ds.rounds; res->windows = ds.windows;
    res->shift_pairs = ds.shift_pairs; res->exceptional = ds.exceptional;
    res->final_blocks = ds.final_blocks; res->launches = be.launches; res->apply_flops = ds.apply_flops;
    res->host_seconds = t_drive;
    if (profile) {
      double ms[6] = {0, 0, 0, 0, 0, 0};
      if (dbg_env("PSD_MS_VERBOSE")) {
        double gaps[36] = {0};
        cudaStreamSynchronize(st);
        be.tm.collect_gaps(gaps);
        fprintf(stderr, "[psd ms gaps, ms] scan->chase %.1f | chase->apply %.1f | apply->scan %.1f | scan->scan %.1f | apply->chase %.1f | other %.1f\n",
                gaps[3 * 6 + 0], gaps[0 * 6 + 1], gaps[1 * 6 + 3], gaps[3 * 6 + 3], gaps[1 * 6 + 0],
                gaps[4 * 6 + 1] + gaps[1 * 6 + 4] + gaps[3 * 6 + 4] + gaps[3 * 6 + 1] + gaps[1 * 6 + 1]);
      }
      be.tm.collect(ms);
      be.tm_far.collect(ms);
      for (int k = 0; k < kShiftSlots; k++) be.tm_side[k].collect(ms);
      res->ms_chase = ms[0]; res->ms_apply = ms[1]; res->ms_shifts = ms[2]; res->ms_scan = ms[3]; res->ms_final = ms[4];
      res->ms_rounds = ms[5];
    }
  }
  if (dprof) {
    long long hp[16];
    cudaMemcpy(hp, dprof, sizeof(hp), cudaMemcpyDeviceToHost);
    cudaFree(dprof);
    const double k = hp[6] ? 1.0 / hp[6] : 0.0;
    fprintf(stderr, "[psd ms chase, CTA 0 of %lld launches, cycles per launch] chain %.0f | columns %.0f | rows %.0f | write-back %.0f | whole CTA %.0f | steps %.1f | scan end -> chase start %.1f us (globaltimer) | -> stamp kernel %.1f us\n",
            hp[6], hp[0] * k, hp[1] * k, hp[2] * k, hp[3] * k, hp[4] * k, hp[5] * k, hp[7] * k * 1e-3, hp[8] * k * 1e-3);
  }
  if (dbg_env("PSD_MS_VERBOSE"))
    fprintf(stderr, "[psd ms] n %d p %d W %d NB %d nsw %d: status %d, %d sets, %lld rounds, %lld windows, %lld pairs, %d exceptional, %d final blocks, %d idle windows, %.3f TFLOP applied; host %.3f s (blocked: scans %.3f, shifts %.3f, plan ring %.3f)\n",
            n, p, g.W, g.NB, cfg.nsw, status, ds.sweeps, ds.rounds, ds.windows, ds.shift_pairs, ds.exceptional,
            ds.final_blocks, idle_windows, ds.apply_flops * 1e-12, t_drive, be.wait_scan, be.wait_shift, be.wait_plan);
  return cudaSuccess;
}

}  // namespace ms
}  // namespace psd
