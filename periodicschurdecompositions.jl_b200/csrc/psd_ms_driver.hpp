// Host driver of the large-N multishift periodic QR iteration (pure C++, no CUDA): the packet
// pipeline, the shift strategy and the window schedule.  It talks to a backend - the CUDA kernels
// (psd_ms.cu) in the product, the CPU emulation of the same kernels in tests/ms_emul/ - so the
// control logic that decides convergence is tested on the CPU as well.
//
// Replaces the outer iteration of pschur!(H1, Hs) (PeriodicSchurDecompositions.jl:442-1060) for
// N >= 192.  Organisation: a continuous pipeline of bulge packets.
//   round      every packet in flight moves down by D rows inside its own diagonal window (chase
//              kernel, one CTA per window), then the off-window parts of H_j and Z_j are updated
//              on the tensor cores, then the subdiagonal of H_1 is scanned for negligible entries
//   blocks     every unreduced diagonal block of order > W the scan reports (the lowest
//              max_blocks of them) is worked on at the same time: the reference finishes the lowest
//              block before it touches the next one, which on the GPU leaves a handful of windows
//              per round for two thirds of the rounds
//   injection  every second round (as soon as the top window of a block is free) a new packet
//              of NB bulges is introduced at the top of that block, so up to N / W packets are
//              in flight and the pipeline never drains between "sweeps"
//   shifts     eigenvalues of the trailing ns x ns block of a block, computed by the
//              reference algorithm on one CTA on a side stream from a snapshot of that block;
//              the supply is free running: a new set is requested every few packets, and a packet
//              takes the newest complete set when it is introduced (chosen on the device), so
//              neither the host nor the main stream ever waits for a shift computation (stale
//              shifts cost little convergence: scripts/ms_proto.py)
//   control    the host plans round r from the scan made after round r - lag (a fixed lag, so the
//              schedule is a deterministic function of the data while the device queue stays
//              full); a packet learns about deflations that happened since it was planned from
//              the exact zeros of its own window (clamp_block_end)
//   finish     all remaining blocks (order <= W) are reduced independently by one CTA each
#pragma once
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <deque>
#include <utility>
#include <vector>

#include "psd_ms_core.cuh"

namespace psd {
namespace ms {

struct DriverStats {
  int sweeps = 0;            // shift sets used
  long long rounds = 0;
  long long windows = 0;     // window-rounds (chase CTAs launched)
  long long shift_pairs = 0; // bulges introduced
  int exceptional = 0;
  int final_blocks = 0;
  double apply_flops = 0.0;  // 2 * wl^2 * (extent) summed over the tensor-core updates
};

struct DriverConfig {
  int n = 0, p = 0;
  int wantT = 1, wantZ = 1;
  int nsw = 12;         // order of the shift window (<= 64, limited by shared memory for large p)
  int rep_max = 2;      // a new shift set is requested after (pairs of a set) x rep_max bulges
  int sets_ahead = 6;   // (unused by the free-running shift supply; kept for the emulation switches)
  int lag = 3;          // rounds between a scan and the plan that uses it
  int shift_blocks = 1; // consecutive shift sets come from this many different trailing diagonal blocks
  int scan_every = 1;   // the subdiagonal is scanned after every scan_every-th round
  long long max_rounds = 0;  // 0: (256 + 100 n / D) maxitfac / 30
  int maxitfac = 30;    // the caller's iteration budget factor (<= 0: 30), scales the round cap
  int max_blocks = 4;   // active diagonal blocks worked on concurrently (1: only the lowest, like the reference)
  int new_block_delay = 4;  // rounds between the first shift request of a new block and its first packet
                            // (its own shift set is then normally complete; measured in profiles/r2_large_n_tuning.md)
};

struct ScanInfo {
  int ilo = 0, ihi = -1, done = 0, nzero = 0;  // lowest active block
  int nb = 0;                                   // active blocks reported (lowest first)
  int blo[MS_MAXBLK] = {0}, bhi[MS_MAXBLK] = {0};
};

struct Packet {
  int s;      // first row of the next window
  int hops;   // rounds done
  int nbul, pair0, npairs, pair_off;
  int ilo, ihi;  // active block when the packet was introduced
  int fin_s;     // position at which the packet was first seen in finished territory (-1: not yet)
  WinDesc last;  // its window of the latest round it took part in (hops > 0)
};

// Shift supply and stagnation counters of one active block.
struct BlockCtl {
  int ilo = 0, ihi = -1;
  int req_lo = -1;        // first source row of the newest shift set requested for it (-1: none)
  int since_request = 0;  // bulges introduced since then
  int quota = 0;          // ... after which the next set is requested
  int idle_sets = 0;      // shift sets requested since the block last changed
  long long ready_round = 0;  // no packet before this round (first shift set still being computed)
  bool seen = false;
};

// status: 0 = reduced to blocks of order <= W and finished; 1 = no convergence (the factors are
// still a valid Hessenberg-triangular form with Z accumulated; the caller may fall back); 2 = the
// drain before status 1 did not end within its bound (factors unusable; the caller reports failure).
//
// Giving up (round cap, stagnation, or two windows of one round that would overlap) drains the
// pipeline first: no new packet, no new shift set, and rounds continue until every packet has
// chased its bulges off the bottom of its block (retire rules below).  The drain plans the lowest
// packet first; a packet whose window would overlap one already planned is held back a round.  A
// held packet still hands the scan its chain (its latest window with T = 0, which the chase and
// update kernels skip), so no deflation is ever made inside one of its bulges.
template <class Backend>
int drive(Backend& be, const DriverConfig& cfg, DriverStats& st) {
  const Geom g = geom_for(cfg.p);
  const int n = cfg.n, W = g.W, D = g.D;
  // the reference's budget is maxitfac * n iterations: the round cap scales with maxitfac / 30 and
  // is 256 + 100 n / D at the default
  const long long maxitfac = cfg.maxitfac > 0 ? cfg.maxitfac : 30;
  const long long max_rounds =
      cfg.max_rounds > 0 ? cfg.max_rounds : std::max(1LL, (256 + 100LL * n / D) * maxitfac / 30);
  // a packet leaves after at most n / D + 1 rounds; one held back behind a lower packet loses at
  // most W / D rounds
  const long long drain_max = (n + W) / D + 4;
  const int lag = std::max(1, cfg.lag);
  const bool trace = be.trace();
  const int max_blocks = std::max(1, std::min(cfg.max_blocks, (int)MS_MAXBLK));

  ScanInfo info;
  be.scan_wait(be.scan_async(nullptr, 0, W), info);
  std::deque<int> scan_tickets;   // scans made after the rounds enqueued so far
  std::vector<Packet> pk;
  std::vector<WinDesc> wins;
  std::vector<BlockCtl> blocks;   // active blocks being worked on (at most max_blocks, lowest first)
  int next_slot = 0;
  long long pair_counter = 0;     // running index of the next shift pair (taken modulo the set size on the device)
  bool any_set = false;
  bool draining = false;
  long long drain_rounds = 0;
  auto start_drain = [&]() {
    draining = true;
    // a packet that has not had its first window yet has not touched the matrix
    pk.erase(std::remove_if(pk.begin(), pk.end(), [](const Packet& q) { return q.hops == 0; }), pk.end());
  };

  // Shift supply: free running.  A request snapshots the trailing part of a block on the main
  // stream and computes its eigenvalues on a side stream; a packet that is introduced takes the
  // newest complete set that was computed from rows of its block (decided on the device; failing
  // that, the newest set of any block), so the host never waits for a shift computation.  `fence`
  // makes the main stream wait for this request (very first set only).
  auto request_set = [&](BlockCtl& b, double perturb, bool fence) {
    const int m = b.ihi - b.ilo + 1;
    int ns = std::min(cfg.nsw, 2 * (m / 3));
    ns = std::max(2, ns & ~1);
    // Many packets are in flight at once; shifts that all approximate the same few eigenvalues
    // would be wasted, so consecutive sets can be the Ritz values of consecutive diagonal blocks
    // of the trailing part of the block (block 0 = the trailing block itself).
    int blk = 0;
    if (cfg.shift_blocks > 1 && !fence) blk = (int)(st.sweeps % cfg.shift_blocks);
    while (blk > 0 && b.ihi - (blk + 1) * ns + 1 < b.ilo) blk--;
    const int lo = b.ihi - (blk + 1) * ns + 1;
    be.shifts_request(next_slot, lo, ns, perturb, fence);
    next_slot = (next_slot + 1) % be.shift_slots();
    b.req_lo = lo;
    b.since_request = 0;
    b.quota = std::max(g.NB, (ns / 2) * std::max(1, cfg.rep_max));
    b.idle_sets++;
    st.sweeps++;
    any_set = true;
    if (trace)
      fprintf(stderr, "[psd ms] shift set %d for block [%d, %d] (%d x %d)%s, %zu packets in flight\n", st.sweeps, b.ilo,
              b.ihi, ns, ns, fence ? " fenced" : "", pk.size());
  };

  for (long long r = 0;; r++) {
    // ---- block information: the scan made `lag` rounds ago ----
    bool fresh = (r == 0);
    while ((int)scan_tickets.size() > lag - 1) {
      be.scan_wait(scan_tickets.front(), info);
      scan_tickets.pop_front();
      fresh = true;
    }
    if (!be.ok()) return 1;
    if (fresh) {
      // match the reported blocks with the ones being worked on: blocks only shrink or split, so a
      // reported block continues the entry that contains it - the part that holds the source rows
      // of the entry's newest shift set inherits the shift supply, other parts start afresh
      std::vector<BlockCtl> next;
      const int nb = info.done ? 0 : std::min(info.nb, max_blocks);
      for (int k = 0; k < nb; k++) {
        BlockCtl e;
        e.ilo = info.blo[k]; e.ihi = info.bhi[k];
        for (const BlockCtl& o : blocks)
          if (e.ilo >= o.ilo && e.ihi <= o.ihi) {
            const bool same = (e.ilo == o.ilo && e.ihi == o.ihi);
            if (o.req_lo >= e.ilo && o.req_lo <= e.ihi) {
              e.req_lo = o.req_lo; e.since_request = o.since_request; e.quota = o.quota;
              e.ready_round = o.ready_round;
            }
            e.idle_sets = (same && info.nzero == 0) ? o.idle_sets : 0;
            break;
          }
        next.push_back(e);
      }
      blocks.swap(next);
    }
    // ---- retire packets that have left the matrix or travel through finished territory ----
    {
      // rows that may still belong to an active block: the reported ones and, when the list may
      // be truncated, everything above the highest reported block
      auto maybe_active = [&](int row) {
        if (info.done) return false;
        for (int k = 0; k < info.nb; k++)
          if (row >= info.blo[k] && row <= info.bhi[k]) return true;
        return info.nb == (int)MS_MAXBLK && row < info.blo[info.nb - 1];
      };
      size_t k = 0;
      for (size_t i = 0; i < pk.size(); i++) {
        // (a) the previous window reached the bottom of the block the packet was planned for
        // (every bulge chased off), or (b) the packet has travelled 2 W rows through finished
        // territory (blocks of order <= W) since it was first seen there: each of its bulges has
        // met an exact zero of the subdiagonal within W + 3 NB rows and has been chased off at it
        // (clamp_block_end)
        Packet& q = pk[i];
        if (q.fin_s < 0 && !maybe_active(q.s)) q.fin_s = q.s;
        const bool gone = (q.hops > 0 && q.s - D + W >= q.ihi + 1) || (q.fin_s >= 0 && q.s >= q.fin_s + 2 * W);
        if (!gone) pk[k++] = q;
      }
      pk.resize(k);
    }
    if (!draining && info.done && pk.empty()) {
      // drain the scans still in flight (they cannot undo `done`: zeros are only ever added)
      ScanInfo tmp;
      while (!scan_tickets.empty()) { be.scan_wait(scan_tickets.front(), tmp); scan_tickets.pop_front(); }
      break;
    }
    if (!draining && r > max_rounds) start_drain();
    for (BlockCtl& b : blocks) {
      if (draining) break;
      const int pass_sets = std::max(1, ((b.ihi - b.ilo + 1) / W) / std::max(1, cfg.nsw / (2 * g.NB)));
      if (b.idle_sets > 60 + 40 * pass_sets) {
        start_drain();
        break;
      }
      // ---- shift sets ----
      const int ex_every = 6 + 4 * pass_sets;  // sets without any deflation before the shifts are spread
      double perturb = 0.0;
      if (b.idle_sets >= ex_every && b.idle_sets % ex_every == 0) perturb = 0.5;  // exceptional shifts
      if (b.req_lo < 0 || b.since_request >= b.quota) {
        if (b.req_lo < 0 && any_set) b.ready_round = r + cfg.new_block_delay;
        request_set(b, perturb, !any_set);
        if (perturb != 0.0) st.exceptional++;
      }
      // ---- introduce a packet when the top window of the block is free ----
      bool top_free = true;
      for (const Packet& q : pk)
        if (q.s < b.ilo + W && q.s + W > b.ilo) top_free = false;
      if (top_free && r >= b.ready_round && (int)pk.size() < be.max_windows()) {
        Packet q;
        q.nbul = g.NB;
        q.pair0 = (int)(pair_counter % 1000000);
        q.npairs = 0;   // the set (and its size) is chosen on the device when the window runs
        q.pair_off = 0;
        q.ilo = b.ilo; q.ihi = b.ihi;
        q.s = b.ilo; q.hops = 0; q.fin_s = -1;
        pair_counter += q.nbul;
        b.since_request += q.nbul;
        st.shift_pairs += q.nbul;
        pk.push_back(q);
      }
    }
    // ---- this round's windows ----
    auto window_of = [&](const Packet& q) {
      WinDesc w;
      w.idle = 0;
      w.ilo = q.ilo; w.ihi = q.ihi; w.nbul = q.nbul; w.pair0 = q.pair0; w.npairs = q.npairs; w.pair_off = q.pair_off;
      if (q.hops == 0) {
        w.intro = 1; w.s = q.ilo; w.kbase = q.ilo - 1; w.T = D + 1 + 3 * (q.nbul - 1);
      } else {
        w.intro = 0; w.s = q.s; w.kbase = q.s + 3 * (q.nbul - 1); w.T = D;
      }
      w.wl = (w.s + W <= q.ihi + 1) ? W : q.ihi + 1 - w.s;
      if (w.s + W >= q.ihi + 1) {
        // last window of this packet: chase every bulge off the bottom
        const int last_base = w.kbase - 3 * (q.nbul - 1);
        w.T = std::max(1, (q.ihi - 2) - last_base + 1);
      }
      return w;
    };
    wins.clear();
    std::vector<char> moves(pk.size(), 1);
    if (!draining) {
      for (const Packet& q : pk) wins.push_back(window_of(q));
      // windows of one round must be disjoint (packets of one block keep their distance by
      // construction; this also covers packets that outlive a split of their block)
      std::vector<std::pair<int, int>> span;
      for (const WinDesc& w : wins) span.emplace_back(w.s, w.s + w.wl);
      std::sort(span.begin(), span.end());
      for (size_t i = 1; i < span.size() && !draining; i++)
        if (span[i].first < span[i - 1].second) start_drain();
    }
    size_t nmove = pk.size();
    if (draining) {
      if (pk.empty()) {
        ScanInfo tmp;
        while (!scan_tickets.empty()) { be.scan_wait(scan_tickets.front(), tmp); scan_tickets.pop_front(); }
        return 1;
      }
      if (++drain_rounds > drain_max) return 2;
      // lowest packet first; one whose window would overlap a window already planned is held back
      std::vector<size_t> order(pk.size());
      for (size_t i = 0; i < pk.size(); i++) order[i] = i;
      std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return pk[a].s > pk[b].s; });
      wins.clear();
      moves.assign(pk.size(), 0);
      std::vector<WinDesc> held;
      for (size_t i : order) {
        const WinDesc w = window_of(pk[i]);
        bool clash = false;
        for (size_t k = 0; k < pk.size(); k++) {
          if (!moves[k]) continue;
          const WinDesc o = window_of(pk[k]);
          clash |= (w.s < o.s + o.wl && o.s < w.s + w.wl);
        }
        if (clash) {
          WinDesc h = pk[i].last;
          h.T = 0;  // chain only: the chase and update kernels skip the window, the scan spares the chain
          held.push_back(h);
        } else {
          moves[i] = 1;
        }
      }
      for (size_t i = 0; i < pk.size(); i++)
        if (moves[i]) wins.push_back(window_of(pk[i]));
      nmove = wins.size();
      wins.insert(wins.end(), held.begin(), held.end());
    }
    for (size_t i = 0, k = 0; i < pk.size(); i++) {
      if (!moves[i]) continue;
      Packet& q = pk[i];
      q.last = wins[k++];
      q.s = (q.hops == 0) ? q.ilo + D : q.s + D;
      q.hops++;
    }
    if (!wins.empty()) {
      be.round(wins);
      st.rounds++;
      st.windows += (long long)nmove;
      for (size_t k = 0; k < nmove; k++) {
        const WinDesc& w = wins[k];
        const double left = (cfg.wantT ? n : w.ihi + 1) - (w.s + w.wl);
        const double right = w.s - (cfg.wantT ? 0 : w.ilo);
        const double z = cfg.wantZ ? n : 0;
        st.apply_flops += 2.0 * w.wl * w.wl * (left + right + z) * cfg.p;
      }
    }
    if (r % std::max(1, cfg.scan_every) == 0) scan_tickets.push_back(be.scan_async(wins.data(), (int)wins.size(), W));
  }
  int nblocks = 0;
  be.finish(nblocks);
  st.final_blocks = nblocks;
  return be.ok() ? 0 : 1;
}

}  // namespace ms
}  // namespace psd
