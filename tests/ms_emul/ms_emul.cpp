// TEST INFRASTRUCTURE ONLY: CPU emulation of the large-N multishift periodic QR iteration.
//
// It compiles the product's own host/device headers (csrc/psd_ms_core.cuh: the in-window bulge
// chase; csrc/psd_ms_driver.hpp: sweep loop, shift strategy, window schedule) with g++ and runs
// them against an emulated backend: a CTA is emulated by calling every (bulge, role) of a phase in
// turn (in an order that changes from phase to phase, which also checks that the phases are
// race-free), the tensor-core window updates by plain loops, and the two places where the CUDA
// path calls periodic_qr_cta (shifts, final blocks) by the CPU oracle's restatement of the same
// reference routine.  Nothing under periodicschurdecompositions.jl_b200/ links or loads this.
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../oracle/psdo_real.hpp"
#include "../../periodicschurdecompositions.jl_b200/csrc/psd_ms_driver.hpp"

using namespace psd::ms;

namespace {

struct HostExec {
  static constexpr int LANES = 1;
  int nb = 0;
  unsigned flip = 0;
  BState st[MS_MAXNB][2];
  template <class F>
  void each(F&& f) {
    // vary the order in which the emulated warps run: a correct phase does not depend on it
    flip = flip * 1103515245u + 12345u;
    const bool rev = (flip >> 16) & 1, rfirst = (flip >> 17) & 1;
    for (int i = 0; i < nb; i++) {
      const int b = rev ? nb - 1 - i : i;
      for (int q = 0; q < 2; q++) {
        const int role = rfirst ? 1 - q : q;
        f(b, role, 0, st[b][role]);
      }
    }
  }
  void barrier() {}
  void tick(int) {}
};

struct EmuBackend {
  int n, p, wantT, wantZ, maxitfac;
  Geom g;
  std::vector<double*> H, Z;
  double* eig;
  int info = 0;
  std::vector<double> U;       // [p][n * W]
  std::vector<double> pairs;
  std::vector<WinDesc> plan;
  long long chase_steps = 0;

  double& h(int j, int r, int c) { return H[j][r + (size_t)c * n]; }

  bool ok() const { return true; }
  int shift_slots() const { return 8; }
  bool trace() const { return getenv("PSD_MS_TRACE") != nullptr; }
  int max_windows() const { return 160; }
  int pair_offset(int slot) const { return slot * 66; }
  std::vector<ScanInfo> scan_ring = std::vector<ScanInfo>(16);
  long long nscan = 0;

  int scan_async(const WinDesc* wins, int cnt, int nmin) {
    const int slot = (int)(nscan++ % 16);
    ScanInfo& out = scan_ring[slot];
    const double smlnum = DBL_MIN * ((double)n / DBL_EPSILON);
    out.nzero = 0;
    std::vector<int> first, last;
    for (int w = 0; w < cnt; w++) {
      int a, b;
      if (chain_after_round(wins[w], g.W, g.D, a, b)) { first.push_back(a); last.push_back(b); }
    }
    for (int k = 1; k < n; k++) {
      bool skip = false;
      for (size_t w = 0; w < first.size(); w++) skip |= (k - 1 >= first[w] && k - 1 <= last[w]);
      if (skip) continue;
      const double sub = h(0, k, k - 1);
      if (sub != 0.0 && ms_negligible(sub, h(0, k - 1, k - 1), h(0, k, k), smlnum)) {
        h(0, k, k - 1) = 0.0;
        out.nzero++;
      }
    }
    // unreduced diagonal blocks of order > nmin, lowest first (as ms_scan_body reports them)
    out.nb = 0;
    for (int k = n - 1; k >= 0;) {
      int r = k;
      while (r > 0 && h(0, r, r - 1) != 0.0) r--;
      if (k - r + 1 > nmin && out.nb < (int)MS_MAXBLK) {
        out.blo[out.nb] = r; out.bhi[out.nb] = k;
        out.nb++;
      }
      k = r - 1;
    }
    out.ilo = out.nb ? out.blo[0] : 0;
    out.ihi = out.nb ? out.bhi[0] : -1;
    out.done = out.nb == 0;
    return slot;
  }
  void scan_wait(int slot, ScanInfo& info) { info = scan_ring[slot]; }

  int slot_pairs[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int slot_seq[8] = {0, 0, 0, 0, 0, 0, 0, 0}, slot_lo[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  int shift_seq = 0;
  void shifts_request(int slot, int lo, int m, double perturb, bool /*fence*/) {
    std::vector<double> buf((size_t)p * m * m);
    std::vector<psdo::Mat> Hm(p), Zm(p);
    for (int j = 0; j < p; j++) {
      Hm[j] = psdo::Mat{buf.data() + (size_t)j * m * m, m};
      const int keep = (j == 0) ? 1 : 0;
      for (int c = 0; c < m; c++)
        for (int r = 0; r < m; r++) buf[(size_t)j * m * m + r + (size_t)c * m] = (r > c + keep) ? 0.0 : h(j, lo + r, lo + c);
    }
    std::vector<double> lre(m), lim(m);
    const int inf = psdo::real_periodic_qr(m, p, Hm, Zm, false, false, 30, lre.data(), lim.data());
    if (pairs.empty()) pairs.assign((size_t)8 * 66 * 4, 0.0);
    if (getenv("MS_EMUL_VERBOSE")) fprintf(stderr, "[emul] shifts slot %d lo %d m %d info %d\n", slot, lo, m, inf);
    slot_pairs[slot] = pair_shifts(lre.data(), lim.data(), inf, m, perturb, pairs.data() + (size_t)pair_offset(slot) * 4);
    // the emulation completes a request at once
    slot_lo[slot] = lo;
    slot_seq[slot] = (slot_pairs[slot] > 0) ? ++shift_seq : 0;
  }


  double* Uptr(int j, int s) { return U.data() + (size_t)j * n * g.W + (size_t)s * g.W; }

  void apply(const WinDesc* wins, int cnt) {
    std::vector<double> tmp(64);
    for (int w = 0; w < cnt; w++) {
      const WinDesc& d = wins[w];
      const int s = d.s, wl = d.wl;
      for (int j = 0; j < p; j++) {
        const double* Uj = Uptr(j, s);
        // left: H_j[s:s+wl, c_lo:c_hi) <- U_j' * .
        const int c_lo = s + wl, c_hi = wantT ? n : d.ihi + 1;
        for (int c = c_lo; c < c_hi; c++) {
          for (int m = 0; m < wl; m++) {
            double acc = 0.0;
            for (int k = 0; k < wl; k++) acc += Uj[k + (size_t)m * wl] * h(j, s + k, c);
            tmp[m] = acc;
          }
          for (int m = 0; m < wl; m++) h(j, s + m, c) = tmp[m];
        }
        // Z_j[:, s:s+wl) <- . * U_j
        if (wantZ)
          for (int r = 0; r < n; r++) {
            for (int c = 0; c < wl; c++) {
              double acc = 0.0;
              for (int k = 0; k < wl; k++) acc += Z[j][r + (size_t)(s + k) * n] * Uj[k + (size_t)c * wl];
              tmp[c] = acc;
            }
            for (int c = 0; c < wl; c++) Z[j][r + (size_t)(s + c) * n] = tmp[c];
          }
      }
    }
    for (int w = 0; w < cnt; w++) {
      const WinDesc& d = wins[w];
      const int s = d.s, wl = d.wl;
      for (int j = 0; j < p; j++) {
        const double* Uj = Uptr(j, s);
        const int jm = (j == 0) ? p - 1 : j - 1;
        const int r_lo = wantT ? 0 : d.ilo;
        for (int r = r_lo; r < s; r++) {
          for (int c = 0; c < wl; c++) {
            double acc = 0.0;
            for (int k = 0; k < wl; k++) acc += h(jm, r, s + k) * Uj[k + (size_t)c * wl];
            tmp[c] = acc;
          }
          for (int c = 0; c < wl; c++) h(jm, r, s + c) = tmp[c];
        }
      }
    }
  }

  long long max_rounds = -1, nrounds = 0, held_windows = 0;
  bool skip_apply = false;
  void round(const std::vector<WinDesc>& wins_) {
    if (max_rounds >= 0 && nrounds >= max_rounds) return;
    nrounds++;
    plan = wins_;
    const int off = 0, cnt = (int)plan.size();
    const int W = g.W, LD = g.LD;
    std::vector<double> Hw((size_t)p * W * LD), Uw((size_t)p * W * LD);
    for (int w = 0; w < cnt; w++) {
      WinDesc& dd = plan[off + w];
      if (dd.T == 0) {  // packet held back: the CUDA chase kernel returns at once
        held_windows++;
        continue;
      }
      if (dd.intro) {  // newest complete shift set of this block, as the CUDA kernel picks it
        int best = -1, bseq = 0, any = -1, aseq = 0;
        for (int k = 0; k < 8; k++) {
          if (slot_seq[k] <= 0) continue;
          if (slot_lo[k] >= dd.ilo && slot_lo[k] <= dd.ihi && slot_seq[k] > bseq) { best = k; bseq = slot_seq[k]; }
          if (slot_seq[k] > aseq) { any = k; aseq = slot_seq[k]; }
        }
        const int sl = best >= 0 ? best : any;
        dd.pair_off = sl >= 0 ? pair_offset(sl) : 0;
        dd.npairs = sl >= 0 ? slot_pairs[sl] : 0;
      }
      const WinDesc& d = dd;
      if (getenv("MS_EMUL_VERBOSE"))
        fprintf(stderr, "[emul] round %lld win s %d wl %d kbase %d nbul %d T %d ilo %d ihi %d pair0 %d/%d intro %d\n", nrounds,
                d.s, d.wl, d.kbase, d.nbul, d.T, d.ilo, d.ihi, d.pair0, d.npairs, d.intro);
      Ctx c;
      c.p = p; c.W = W; c.LD = LD; c.Hw = Hw.data(); c.Uw = Uw.data(); c.shifts = pairs.data(); c.d = d;
      for (int j = 0; j < p; j++)
        for (int cc = 0; cc < d.wl; cc++)
          for (int r = 0; r < d.wl; r++) {
            c.H(j + 1)[r + (size_t)cc * LD] = h(j, d.s + r, d.s + cc);
            c.U(j + 1)[r + (size_t)cc * LD] = (r == cc) ? 1.0 : 0.0;
          }
      int bihi[MS_MAXNB];
      c.bihi = bihi;
      std::vector<double> mbox((size_t)MS_MAXNB * MS_MAXP * MB_STRIDE, 0.0);
      c.mbox = mbox.data();
      for (int b = 0; b < d.nbul; b++) bihi[b] = clamp_block_end(c, b);
      HostExec ex;
      ex.nb = g.NB;
      for (int b = 0; b < g.NB; b++)
        for (int q = 0; q < 2; q++) ex.st[b][q].active = 0;
      chase_window(c, ex);
      chase_steps += (long long)d.T * d.nbul;
      if (getenv("MS_EMUL_VERBOSE")) {
        int bad = 0;
        for (int j = 0; j < p; j++)
          for (int cc = 0; cc < d.wl; cc++)
            for (int r = 0; r < d.wl; r++) {
              if (!std::isfinite(c.H(j + 1)[r + (size_t)cc * LD])) { if (!bad) fprintf(stderr, "[emul] non-finite H_%d(%d,%d) win s %d\n", j + 1, r, cc, d.s); bad++; }
              if (!std::isfinite(c.U(j + 1)[r + (size_t)cc * LD])) { if (!bad) fprintf(stderr, "[emul] non-finite U_%d(%d,%d) win s %d\n", j + 1, r, cc, d.s); bad++; }
            }
      }
      if (getenv("MS_EMUL_COUNTID")) {
        bool ident = true;
        for (int j = 0; j < p && ident; j++)
          for (int cc = 0; cc < d.wl && ident; cc++)
            for (int r = 0; r < d.wl; r++)
              if (c.U(j + 1)[r + (size_t)cc * LD] != ((r == cc) ? 1.0 : 0.0)) { ident = false; break; }
        static long long nid = 0, nall = 0;
        nall++;
        nid += ident;
        if (nall % 500 == 0) fprintf(stderr, "[emul] identity windows %lld of %lld\n", nid, nall);
      }
      if (getenv("MS_EMUL_DUMPU") && nrounds == atoi(getenv("MS_EMUL_DUMPU"))) {
        // zero pattern of the accumulated window transformations in 4 x 8 blocks (k-step x fragment)
        for (int j = 0; j < p; j++) {
          fprintf(stderr, "[emul] U_%d of window s %d wl %d intro %d T %d (rows = k in steps of 4, columns in steps of 8; . = all zero)\n", j + 1, d.s, d.wl, d.intro, d.T);
          for (int k0 = 0; k0 < d.wl; k0 += 4) {
            for (int m0 = 0; m0 < d.wl; m0 += 8) {
              bool nzb = false;
              for (int k = k0; k < std::min(d.wl, k0 + 4); k++)
                for (int m = m0; m < std::min(d.wl, m0 + 8); m++) nzb |= (c.U(j + 1)[k + (size_t)m * LD] != 0.0);
              fputc(nzb ? '#' : '.', stderr);
            }
            fputc('\n', stderr);
          }
        }
      }
      for (int j = 0; j < p; j++) {
        double* ud = Uptr(j, d.s);
        for (int cc = 0; cc < d.wl; cc++)
          for (int r = 0; r < d.wl; r++) {
            h(j, d.s + r, d.s + cc) = c.H(j + 1)[r + (size_t)cc * LD];
            ud[r + (size_t)cc * d.wl] = c.U(j + 1)[r + (size_t)cc * LD];
          }
      }
    }
    std::vector<WinDesc> moved;  // (held-back packets have no update)
    for (const WinDesc& d : plan)
      if (d.T != 0) moved.push_back(d);
    apply(moved.data(), (int)moved.size());
  }

  double junk = 0.0;  // largest entry below the Hessenberg / triangular structure when the pipeline ends
  void finish(int& nblocks) {
    nblocks = 0;
    for (int j = 0; j < p; j++)
      for (int c = 0; c < n; c++)
        for (int r = c + (j == 0 ? 2 : 1); r < n; r++) junk = std::max(junk, std::fabs(h(j, r, c)));
    if (max_rounds >= 0) return;
    std::vector<WinDesc> list;
    for (int k = 0; k < n;) {
      int e = k;
      while (e + 1 < n && h(0, e + 1, e) != 0.0) e++;
      const int m = e - k + 1;
      if (m == 1) {
        double l = 1.0;
        for (int j = 0; j < p; j++) l *= h(j, k, k);
        eig[2 * k] = l;
        eig[2 * k + 1] = 0.0;
      } else {
        WinDesc d{};
        d.s = k; d.wl = m; d.ilo = k; d.ihi = e; d.npairs = 1;
        list.push_back(d);
      }
      k = e + 1;
    }
    nblocks = (int)list.size();
    const bool vec = wantT || wantZ;
    for (const WinDesc& d : list) {
      const int m = d.wl, s = d.s;
      std::vector<double> hb((size_t)p * m * m), zb((size_t)p * m * m, 0.0);
      std::vector<psdo::Mat> Hm(p), Zm(p);
      for (int j = 0; j < p; j++) {
        Hm[j] = psdo::Mat{hb.data() + (size_t)j * m * m, m};
        Zm[j] = psdo::Mat{zb.data() + (size_t)j * m * m, m};
        const int keep = (j == 0) ? 1 : 0;
        for (int c = 0; c < m; c++)
          for (int r = 0; r < m; r++) {
            hb[(size_t)j * m * m + r + (size_t)c * m] = (r > c + keep) ? 0.0 : h(j, s + r, s + c);
            if (r == c) zb[(size_t)j * m * m + r + (size_t)c * m] = 1.0;
          }
      }
      std::vector<double> lre(m), lim(m);
      const int inf = psdo::real_periodic_qr(m, p, Hm, Zm, vec, vec, maxitfac, lre.data(), lim.data());
      if (inf != 0 && s + inf > info) info = s + inf;
      for (int k = 0; k < m; k++) {
        eig[2 * (s + k)] = lre[k];
        eig[2 * (s + k) + 1] = lim[k];
      }
      if (vec)
        for (int j = 0; j < p; j++) {
          double* ud = Uptr(j, s);
          for (int c = 0; c < m; c++)
            for (int r = 0; r < m; r++) {
              h(j, s + r, s + c) = hb[(size_t)j * m * m + r + (size_t)c * m];
              ud[r + (size_t)c * m] = zb[(size_t)j * m * m + r + (size_t)c * m];
            }
        }
    }
    if (vec && !list.empty()) apply(list.data(), (int)list.size());
  }
};

}  // namespace

extern "C" {

// H: [p][n*n] column-major Hessenberg-triangular factors (rightwards order), Z: [p][n*n] preset
// Schur vectors or NULL.  maxitfac: the caller's budget factor (<= 0: 30).  max_rounds > 0 caps the
// driver's rounds (DriverConfig::max_rounds; the backend keeps working, so a give-up drains).
// stats[10]: sweeps, rounds, windows, shift pairs, exceptional, final blocks, bulge steps, status,
// 1 if a bulge was left behind when the pipeline finished, windows held back by the drain.
// Returns the status of the driver (0 = finished).
int ms_emul_run(int n, int p, double* Hbuf, double* Zbuf, int wantT, int wantZ, int nsw, int rep_max,
                int maxitfac, long long max_rounds, double* eig, int* info, long long* stats) {
  EmuBackend be;
  be.n = n; be.p = p; be.wantT = wantT; be.wantZ = (wantZ && Zbuf) ? 1 : 0;
  be.maxitfac = maxitfac > 0 ? maxitfac : 30;
  be.g = geom_for(p);
  for (int j = 0; j < p; j++) {
    be.H.push_back(Hbuf + (size_t)j * n * n);
    be.Z.push_back(Zbuf ? Zbuf + (size_t)j * n * n : nullptr);
  }
  be.eig = eig;
  be.U.assign((size_t)p * n * be.g.W, 0.0);
  DriverConfig cfg;
  cfg.n = n; cfg.p = p; cfg.wantT = wantT; cfg.wantZ = be.wantZ;
  if (nsw > 0) cfg.nsw = nsw;
  if (rep_max > 0) cfg.rep_max = rep_max;
  cfg.maxitfac = maxitfac;
  if (max_rounds > 0) cfg.max_rounds = max_rounds;
  if (const char* ev = getenv("MS_EMUL_MAXROUNDS")) {
    be.max_rounds = atoll(ev);
    cfg.max_rounds = be.max_rounds + 4;
  }
  if (const char* ev = getenv("MS_EMUL_LAG")) cfg.lag = atoi(ev);
  if (const char* ev = getenv("MS_EMUL_MAXBLOCKS")) cfg.max_blocks = atoi(ev);
  if (const char* ev = getenv("MS_EMUL_BLOCKS")) cfg.shift_blocks = atoi(ev);
  if (const char* ev = getenv("MS_EMUL_AHEAD")) cfg.sets_ahead = atoi(ev);
  DriverStats ds;
  const int status = drive(be, cfg, ds);
  *info = (status == 2) ? n : be.info;  // as psd_ms.cu reports a drain that did not end
  if (stats) {
    stats[0] = ds.sweeps; stats[1] = ds.rounds; stats[2] = ds.windows; stats[3] = ds.shift_pairs;
    stats[4] = ds.exceptional; stats[5] = ds.final_blocks; stats[6] = be.chase_steps; stats[7] = status;
    stats[8] = (be.junk != 0.0) ? 1 : 0;
    stats[9] = be.held_windows;
  }
  return status;
}

void ms_emul_geom(int p, int* out) {
  const Geom g = geom_for(p);
  out[0] = g.W; out[1] = g.D; out[2] = g.NB; out[3] = g.LD;
}

}  // extern "C"
