// Pass scheduler (pure host C++, no CUDA): turns the instruction list of a
// circuit (/root/reference/src/circuit.rs:53-68) into a PLAN -- the sequence of
// passes the executor runs.  The reference has no counterpart: it issues one
// kernel per instruction in program order (src/circuit.rs:175, 226, 278).
//
// What the plan may change, and why it is exact:
//  * Gates acting on disjoint qubits commute as operators, and the reverse-mode
//    quantities of a gate (pre-gate state, post-gate adjoint) are invariant
//    under moving a disjoint gate across it (DESIGN.md "Reordering").  So gates
//    may be re-ordered within the dependency DAG defined by shared qubits.
//  * Density instructions are full barriers (a Diff density must see exactly
//    the gates that precede it in program order, otherwise the gradients of
//    non-unitary directions change).  A k-qubit density (kind class 5) needs
//    all its k qubits local at once.  So does a k-qubit gate (class 6, step
//    ST_GATE_K), which is a full barrier too: nothing is reordered across it.
//    A diagonal k-qubit gate (class 7, step ST_DIAG_K) is a full barrier as
//    well, but like the two-qubit diagonal it needs no local qubit: its rank
//    bits only select entries, so it never causes a remap.
//
// Sharding: with 2^g ranks the top g PHYSICAL bit positions are the rank
// index ("global").  A logical->physical qubit map is maintained; dense gates
// and densities need all their qubits on local positions, diagonal gates do
// not.  When nothing more can run, global qubits are swapped with the local
// qubits whose next use is farthest away (one half-shard exchange per swapped
// pair), which for 1-D brickwork yields the light-cone ("diamond") schedule.
//
// Tiling: consecutive runnable local gates are grouped into TILE passes: a set
// of at most T physical bit positions (always containing the low L bits, for
// coalescing) such that every gate of the pass acts inside the set; the
// executor then streams the state once for the whole group.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <vector>

namespace qdc {

enum StepType : int { ST_GATE = 0, ST_DENS = 1, ST_SWAP = 2, ST_TILE = 3, ST_GATE_K = 4, ST_DIAG_K = 5 };

struct Step {
  int type = ST_GATE;
  int inst = -1;          // GATE / DENS: instruction index
  int p2 = -1, p1 = -1;   // GATE / DENS: physical positions at execution time (p1 = -1: one-qubit)
  int gbit = -1, lpos = -1;  // SWAP: global bit index (physical position n_loc + gbit) <-> local position
  int first = 0, count = 0;  // TILE: range in Plan::tile_steps
  int tb_first = 0, tb_count = 0;  // TILE: range in Plan::tile_bits (sorted physical positions)
  int grp_first = 0, grp_count = 0;  // TILE: range in Plan::groups (register-block groups)
  int nk = 0, pk[6] = {-1, -1, -1, -1, -1, -1};  // k-qubit DENS / GATE_K / DIAG_K (p2 = p1 = -1): physical positions, most significant first
};

// Steps nothing may be moved across: densities and k-qubit gates, dense or diagonal.  (A k-qubit gate has
// p2 = p1 = -1, so it marks no position dirty: treated as an ordinary deferred step, later gates on its qubits could
// overtake it.)
inline bool is_wall(const Step& st) { return st.type == ST_DENS || st.type == ST_GATE_K || st.type == ST_DIAG_K; }

// A register-block group inside a tile pass: `count` consecutive tile gates
// (starting at Plan::tile_steps[first]) that all act within <= 4 positions.
struct Group {
  int first = 0, count = 0;
  int nbits = 0;
  int bits[4] = {-1, -1, -1, -1};  // physical positions, ascending
};

struct Plan {
  std::vector<Step> steps;
  std::vector<Step> tile_steps;   // GATE steps belonging to TILE passes
  std::vector<int> tile_bits;
  std::vector<Group> groups;
  std::vector<int> final_map;     // logical qubit -> physical position after the plan
  bool ok = true;                 // false: some instructions could not be scheduled (plan is truncated)
};

struct SchedInst {
  int kind_class;  // 0: dense q1, 1: dense q2, 2: diagonal q2, 3: density q1, 4: density q2, 5: density on nq qubits,
                   // 6: gate on nq qubits, 7: diagonal gate on nq qubits
  int q2, q1;      // logical qubits (q1 = -1 for one-qubit instructions; both -1 for classes 5, 6 and 7)
  bool skip;       // densities that this sweep does not evaluate
  int nq = 0;      // classes 5, 6 and 7: the logical qubits qk[0..nq-1], most significant first
  int qk[6] = {-1, -1, -1, -1, -1, -1};
};

struct SchedOptions {
  int n = 0;         // total (logical) qubits
  int n_loc = 0;     // local physical positions per rank (n - g)
  int tile_bits = 0; // T: 0 disables tiling
  int low_bits = 0;  // L: low physical positions forced into every tile
  int min_tile_gates = 2;  // a tile pass must hold at least this many gates to beat streaming
  int max_tile_gates = 24; // capacity of the backward tile kernel's parameter block
  int group_bits = 4;      // register-block width: gates of a pass are grouped by <= this many positions
  // Remap victims are taken from physical positions >= swap_min_pos when any such qubit is less urgent
  // than the global one: the exchanged halves then interleave in runs of 2^pos amplitudes, and the
  // measured exchange rate over NVLink (profiles/r1_exchange_bench_2gpu.txt) is 695 GB/s per direction
  // for pos >= 4 (128-byte runs) against 320-510 GB/s for pos 0..3.  0 = pure farthest-next-use choice.
  int swap_min_pos = 4;
  // Tiling strategy: 1 = grow each tile as a window around a seed gate (a gate joins only when it needs no new
  // position; when nothing more fits, the candidate needing the fewest new positions, closest to the window,
  // is admitted) -- light-cone triangles / diamonds over contiguous qubits; 2 = the same with a look-ahead
  // (the candidate that lets the most gates in per new position); 0 = first-fit in program order
  // (scatters a tile's positions over unrelated pairs: 7.5 gates per pass on 32-qubit brickwork against
  // ~2x that for windows).
  int tile_strategy = 2;
};

class Scheduler {
 public:
  Scheduler(const std::vector<SchedInst>& insts, const SchedOptions& opt) : in_(insts), o_(opt) {}

  Plan run() {
    Plan plan;
    const int N = (int)in_.size();
    done_.assign(N, false);
    map_.resize(o_.n);
    for (int q = 0; q < o_.n; q++) map_[q] = q;
    int remaining = 0;
    for (int i = 0; i < N; i++) {
      if (in_[i].skip) done_[i] = true; else remaining++;
    }
    while (remaining > 0) {
      std::vector<Step> ready;
      collect_ready(ready);
      if (!ready.empty()) {
        remaining -= (int)ready.size();
        emit(plan, ready);
        continue;
      }
      // nothing runnable: bring needed global qubits onto local positions
      if (!remap(plan)) {  // e.g. a dense two-qubit gate with a single local position: never placeable
        plan.ok = false;
        break;
      }
    }
    plan.final_map = map_;
    return plan;
  }

 private:
  const std::vector<SchedInst>& in_;
  SchedOptions o_;
  std::vector<bool> done_;
  std::vector<int> map_;  // logical -> physical

  bool is_barrier(const SchedInst& s) const { return s.kind_class >= 3; }   // densities and k-qubit gates (dense, diagonal)
  bool local(int q) const { return map_[q] < o_.n_loc; }

  // One sweep in program order: every instruction whose predecessors (on its
  // qubits) are done and whose placement allows it to run now.
  void collect_ready(std::vector<Step>& ready) {
    const int N = (int)in_.size();
    std::vector<bool> blocked(o_.n, false);
    bool any_blocked = false;
    for (int i = 0; i < N; i++) {
      if (done_[i]) continue;
      const SchedInst& s = in_[i];
      if (is_barrier(s)) {
        // barrier: runs only if everything before it is done
        if (any_blocked) break;
        bool ok = s.nq > 0 || (local(s.q2) && (s.q1 < 0 || local(s.q1)));
        if (s.kind_class != 7)   // a diagonal k-qubit gate runs wherever its qubits are
          for (int j = 0; j < s.nq; j++) ok = ok && local(s.qk[j]);
        if (!ok) break;
        ready.push_back(make_step(i, s.kind_class == 7 ? ST_DIAG_K : s.kind_class == 6 ? ST_GATE_K : ST_DENS));
        done_[i] = true;
        continue;
      }
      const bool dep = blocked[s.q2] || (s.q1 >= 0 && blocked[s.q1]);
      const bool placed = s.kind_class == 2 || (local(s.q2) && (s.q1 < 0 || local(s.q1)));
      if (!dep && placed) {
        ready.push_back(make_step(i, ST_GATE));
        done_[i] = true;
      } else {
        blocked[s.q2] = true;
        if (s.q1 >= 0) blocked[s.q1] = true;
        any_blocked = true;
      }
    }
  }

  Step make_step(int i, int type) const {
    Step st;
    st.type = type;
    st.inst = i;
    if (in_[i].nq > 0) {
      st.nk = in_[i].nq;
      for (int j = 0; j < st.nk; j++) st.pk[j] = map_[in_[i].qk[j]];
      return st;
    }
    st.p2 = map_[in_[i].q2];
    st.p1 = in_[i].q1 >= 0 ? map_[in_[i].q1] : -1;
    return st;
  }

  // ------------------------------------------------------------- tiling
  bool tileable(const Step& st) const {
    return st.type == ST_GATE && st.p2 < o_.n_loc && (st.p1 < 0 || st.p1 < o_.n_loc);
  }

  void emit(Plan& plan, const std::vector<Step>& ready) {
    if (o_.tile_bits <= 0) {
      for (const Step& st : ready) plan.steps.push_back(st);
      return;
    }
    // Greedy grouping in the given (dependency-respecting) order.  A gate may
    // join the open tile if the union of bit sets still fits; a gate that does
    // not fit closes the tile only if it shares a qubit with a gate already
    // deferred... to stay exact and simple we keep strict order: a non-fitting
    // gate is deferred to the next tile together with everything that depends
    // on it (tracked per physical position).
    std::vector<Step> pending(ready.begin(), ready.end());
    while (!pending.empty()) {
      std::vector<int> bits;  // high bits (>= low_bits) of the open tile
      std::vector<Step> in_tile, deferred;
      const int cap = o_.tile_bits - o_.low_bits;
      if (o_.tile_strategy >= 1) {
        if (!tileable(pending[0])) {  // a density / global-diagonal at the head runs on its own
          plan.steps.push_back(pending[0]);
          pending.erase(pending.begin());
          continue;
        }
        grow_window(pending, cap, bits, in_tile, deferred);
      } else {
      std::vector<bool> dirty(o_.n, false);  // positions touched by a deferred step
      for (const Step& st : pending) {
        bool dep = false;
        auto touches = [&](int p) { return p >= 0 && p < o_.n && dirty[p]; };
        if (touches(st.p2) || touches(st.p1)) dep = true;
        bool fits = false;
        if (!dep && tileable(st) && (int)in_tile.size() < o_.max_tile_gates) {
          int extra = 0;
          auto need = [&](int p) {
            if (p < 0 || p < o_.low_bits) return;
            if (std::find(bits.begin(), bits.end(), p) == bits.end()) extra++;
          };
          need(st.p2);
          if (st.p1 != st.p2) need(st.p1);
          if ((int)bits.size() + extra <= cap) {
            fits = true;
            auto add = [&](int p) {
              if (p < 0 || p < o_.low_bits) return;
              if (std::find(bits.begin(), bits.end(), p) == bits.end()) bits.push_back(p);
            };
            add(st.p2);
            add(st.p1);
          }
        }
        if (fits) {
          in_tile.push_back(st);
        } else if (!dep && !tileable(st) && in_tile.empty() && deferred.empty()) {
          // a non-tileable step (density, global-diagonal) at the head runs on its own
          plan.steps.push_back(st);
        } else {
          deferred.push_back(st);
          if (is_wall(st)) {
            // densities and k-qubit gates are barriers: nothing after them may be pulled forward
            for (int p = 0; p < o_.n; p++) dirty[p] = true;
          } else {
            if (st.p2 >= 0) dirty[st.p2] = true;
            if (st.p1 >= 0) dirty[st.p1] = true;
          }
        }
      }
      }
      if ((int)in_tile.size() >= o_.min_tile_gates) {
        Step t;
        t.type = ST_TILE;
        t.first = (int)plan.tile_steps.size();
        t.count = (int)in_tile.size();
        t.grp_first = (int)plan.groups.size();
        group_tile(plan, in_tile);  // appends the gates to plan.tile_steps in group order
        t.grp_count = (int)plan.groups.size() - t.grp_first;
        std::sort(bits.begin(), bits.end());
        t.tb_first = (int)plan.tile_bits.size();
        for (int l = 0; l < o_.low_bits; l++) plan.tile_bits.push_back(l);
        for (int b : bits) plan.tile_bits.push_back(b);
        t.tb_count = (int)plan.tile_bits.size() - t.tb_first;
        plan.steps.push_back(t);
      } else {
        for (const Step& st : in_tile) plan.steps.push_back(st);
      }
      pending.swap(deferred);
    }
  }

  // Window growth (tile_strategy 1).  `pending` is in dependency-respecting order and starts with a
  // tileable gate.  A gate may be chosen only if no earlier, still unchosen step shares a position with it
  // (densities block everything behind them), so the chosen set -- kept in pending order -- is a valid
  // prefix-closed selection and the rest can run afterwards in its original order.
  void grow_window(const std::vector<Step>& pending, int cap, std::vector<int>& bits, std::vector<Step>& in_tile,
                   std::vector<Step>& deferred) {
    grow_window(pending, cap, o_.low_bits, o_.max_tile_gates, bits, in_tile, deferred);
  }

  // Number of still unchosen gates a window over `wbits` would admit (closure under the admission rule).
  int closure_gain(const std::vector<Step>& pending, const std::vector<char>& chosen0, const std::vector<int>& wbits,
                   int free_below, int limit) const {
    const int M = (int)pending.size();
    std::vector<char> chosen(chosen0), dirty(o_.n);
    auto has = [&](int p) { return p < 0 || p < free_below || std::find(wbits.begin(), wbits.end(), p) != wbits.end(); };
    int gain = 0;
    for (bool progress = true; progress && gain < limit;) {
      progress = false;
      std::fill(dirty.begin(), dirty.end(), 0);
      for (int k = 0; k < M && gain < limit; k++) {
        if (chosen[k]) continue;
        const Step& st = pending[k];
        if (!tileable(st)) {
          if (is_wall(st)) break;
          if (st.p2 >= 0 && st.p2 < o_.n) dirty[st.p2] = 1;
          if (st.p1 >= 0 && st.p1 < o_.n) dirty[st.p1] = 1;
          continue;
        }
        const bool dep = dirty[st.p2] || (st.p1 >= 0 && dirty[st.p1]);
        if (!dep && has(st.p2) && has(st.p1)) {
          chosen[k] = 1;
          gain++;
          progress = true;
        } else {
          dirty[st.p2] = 1;
          if (st.p1 >= 0) dirty[st.p1] = 1;
        }
      }
    }
    return gain;
  }

  // `free_below`: positions below it are always available (the tile's forced low positions) and do not count.
  void grow_window(const std::vector<Step>& pending, int cap, int free_below, int max_gates, std::vector<int>& bits,
                   std::vector<Step>& in_tile, std::vector<Step>& deferred) {
    const int M = (int)pending.size();
    std::vector<char> chosen(M, 0);
    int nchosen = 0;
    auto has = [&](int p) { return p < 0 || p < free_below || std::find(bits.begin(), bits.end(), p) != bits.end(); };
    auto extra_of = [&](const Step& st) { return (has(st.p2) ? 0 : 1) + ((st.p1 == st.p2 || has(st.p1)) ? 0 : 1); };
    std::vector<char> dirty(o_.n);
    struct Cand { int k, extra, dist; };
    std::vector<Cand> cands;
    for (;;) {
      // sweep: admit everything that needs no new position; remember the best candidate that does
      bool progress = false;
      int best = -1, best_extra = 0, best_dist = 0;
      cands.clear();
      std::fill(dirty.begin(), dirty.end(), 0);
      bool wall = false;  // a density / non-tileable step ahead blocks everything behind it
      for (int k = 0; k < M && !wall && nchosen < max_gates; k++) {
        if (chosen[k]) continue;
        const Step& st = pending[k];
        if (!tileable(st)) {
          if (is_wall(st)) { wall = true; break; }
          if (st.p2 >= 0 && st.p2 < o_.n) dirty[st.p2] = 1;
          if (st.p1 >= 0 && st.p1 < o_.n) dirty[st.p1] = 1;
          continue;
        }
        const bool dep = dirty[st.p2] || (st.p1 >= 0 && dirty[st.p1]);
        const int extra = dep ? 0 : extra_of(st);
        if (!dep && extra == 0) {
          chosen[k] = 1;
          nchosen++;
          progress = true;
          continue;
        }
        if (!dep && (int)bits.size() + extra <= cap) {
          int dist = 0;  // distance of the gate's new positions from the window (0 for the seed)
          if (!bits.empty()) {
            dist = 1 << 20;
            for (int p : {st.p2, st.p1}) {
              if (p < 0 || has(p)) continue;
              for (int b : bits) dist = std::min(dist, std::abs(p - b));
            }
          }
          if (best < 0 || extra < best_extra || (extra == best_extra && dist < best_dist)) {
            best = k;
            best_extra = extra;
            best_dist = dist;
          }
          if (o_.tile_strategy >= 2) cands.push_back(Cand{k, extra, dist});
        }
        dirty[st.p2] = 1;
        if (st.p1 >= 0) dirty[st.p1] = 1;
      }
      if (progress) continue;  // newly admitted gates may have unblocked others
      if (best < 0 || nchosen >= max_gates) break;
      if (o_.tile_strategy >= 2 && cands.size() > 1) {
        // look-ahead: admit the candidate whose positions let the most gates in per new position
        // (grows a window towards fresh work instead of into qubits that are already ahead in time)
        std::sort(cands.begin(), cands.end(), [](const Cand& a, const Cand& b) {
          return a.dist != b.dist ? a.dist < b.dist : a.k < b.k;
        });
        if (cands.size() > 8) cands.resize(8);
        double best_score = -1;
        for (const Cand& c : cands) {
          std::vector<int> trial = bits;
          const Step& cs = pending[c.k];
          if (!has(cs.p2)) trial.push_back(cs.p2);
          if (!has(cs.p1) && cs.p1 != cs.p2) trial.push_back(cs.p1);
          const int gain = closure_gain(pending, chosen, trial, free_below, max_gates - nchosen);
          const double score = (double)gain / c.extra;
          if (score > best_score + 1e-9) {
            best_score = score;
            best = c.k;
          }
        }
      }
      const Step& st = pending[best];
      if (!has(st.p2)) bits.push_back(st.p2);
      if (!has(st.p1)) bits.push_back(st.p1);
      chosen[best] = 1;
      nchosen++;
    }
    for (int k = 0; k < M; k++) (chosen[k] ? in_tile : deferred).push_back(pending[k]);
  }

  // Second-level grouping for register blocking: partition the gates of one
  // tile pass (in dependency order) into groups acting within <= group_bits
  // positions, deferring what does not fit together with its dependants.
  void group_tile(Plan& plan, const std::vector<Step>& gates) {
    std::vector<Step> pending(gates.begin(), gates.end());
    const int RB = o_.group_bits < 2 ? 2 : (o_.group_bits > 4 ? 4 : o_.group_bits);
    while (!pending.empty()) {
      std::vector<int> bits;
      std::vector<Step> grp, deferred;
      std::vector<bool> dirty(o_.n, false);
      if (o_.tile_strategy >= 1) {
        // same window growth as for the tiles: 3.6 instead of 3.0 gates per register block on brickwork
        grow_window(pending, RB, 0, 1 << 30, bits, grp, deferred);
        pending.clear();
      }
      for (const Step& st : pending) {
        const bool dep = dirty[st.p2] || (st.p1 >= 0 && dirty[st.p1]);
        bool fits = false;
        if (!dep) {
          int extra = 0;
          if (std::find(bits.begin(), bits.end(), st.p2) == bits.end()) extra++;
          if (st.p1 >= 0 && st.p1 != st.p2 && std::find(bits.begin(), bits.end(), st.p1) == bits.end()) extra++;
          if ((int)bits.size() + extra <= RB) {
            fits = true;
            if (std::find(bits.begin(), bits.end(), st.p2) == bits.end()) bits.push_back(st.p2);
            if (st.p1 >= 0 && std::find(bits.begin(), bits.end(), st.p1) == bits.end()) bits.push_back(st.p1);
          }
        }
        if (fits) {
          grp.push_back(st);
        } else {
          deferred.push_back(st);
          dirty[st.p2] = true;
          if (st.p1 >= 0) dirty[st.p1] = true;
        }
      }
      Group g;
      g.first = (int)plan.tile_steps.size();
      g.count = (int)grp.size();
      std::sort(bits.begin(), bits.end());
      g.nbits = (int)bits.size();
      for (int k = 0; k < g.nbits; k++) g.bits[k] = bits[k];
      for (const Step& st : grp) plan.tile_steps.push_back(st);
      plan.groups.push_back(g);
      pending.swap(deferred);
    }
  }

  // --------------------------------------------------------------- remap
  // index (program order) of the first unfinished instruction using qubit q
  std::vector<int> next_use() const {
    const int N = (int)in_.size();
    std::vector<int> nu(o_.n, N + 1);
    for (int i = N - 1; i >= 0; i--) {
      if (done_[i] || in_[i].kind_class == 7) continue;   // a diagonal k-qubit gate needs none of its qubits local
      // (the qubits of a k-qubit density or gate share one next use: a remap for it never evicts another of them,
      // the victims must be strictly less urgent)
      for (int j = 0; j < in_[i].nq; j++) nu[in_[i].qk[j]] = i;
      if (in_[i].nq > 0) continue;
      nu[in_[i].q2] = i;
      if (in_[i].q1 >= 0) nu[in_[i].q1] = i;
    }
    return nu;
  }

  bool remap(Plan& plan) {
    if (o_.n_loc >= o_.n) return false;
    const std::vector<int> nu = next_use();
    std::vector<int> globals, locals;
    for (int q = 0; q < o_.n; q++) (local(q) ? locals : globals).push_back(q);
    std::sort(globals.begin(), globals.end(), [&](int a, int b) { return nu[a] < nu[b]; });  // most urgent first
    const int min_pos = std::min(o_.swap_min_pos, std::max(0, o_.n_loc - 1));
    std::sort(locals.begin(), locals.end(), [&](int a, int b) {
      const bool la = map_[a] < min_pos, lb = map_[b] < min_pos;
      if (la != lb) return lb;                   // positions with short runs last (slow exchanges)
      if (nu[a] != nu[b]) return nu[a] > nu[b];  // least urgent first
      return map_[a] > map_[b];                  // prefer high positions (cheaper, contiguous halves)
    });
    bool any = false;
    std::vector<char> used(locals.size(), 0);
    for (size_t k = 0; k < globals.size(); k++) {
      const int G = globals[k];
      int pick = -1;  // first unused local (in preference order) that is less urgent than G
      for (size_t j = 0; j < locals.size(); j++)
        if (!used[j] && nu[G] < nu[locals[j]]) {
          pick = (int)j;
          break;
        }
      if (pick < 0) break;
      used[pick] = 1;
      const int L = locals[pick];
      Step st;
      st.type = ST_SWAP;
      st.gbit = map_[G] - o_.n_loc;
      st.lpos = map_[L];
      plan.steps.push_back(st);
      std::swap(map_[G], map_[L]);
      any = true;
    }
    return any;
  }
};

// ---- choice of the remap victims' lowest position by a cost model ------------------------------------------------
// Victims at positions >= 4 exchange at the full NVLink rate, but on a qubit chain they cut an island off the low end of
// the register (35-qubit brickwork on 8 ranks with 6-position windows: 205 passes instead of 189, 28 of them with <= 6
// gates); victims from position 2 upwards keep the windows whole and pay with 32-byte runs in the exchange.  Both are
// cheap to plan, so the executor plans every candidate and keeps the cheapest under this model (times in ms at the
// scale of a 2^32-amplitude f32 shard on a B200; only their ratios matter):
struct CostModel {
  double tile_ms = 280;       // one fused pass, forward + reverse (tensor-core blocks: 59)
  double gate_ms = 35;        // one streamed gate, forward + reverse
  double shard_ms = 49.4;     // one full shard over NVLink at 695 GB/s per direction
  int amp_bytes = 8;
  int vec_log2 = 1;           // merged exchanges need positions >= this (circuit.cuh: multi_swap_ok)
  bool merged = true;         // runs of swaps execute as one exchange (k_peer_multiswap)
  // rate relative to 695 GB/s against the length of the contiguous runs: profiles/r1_exchange_bench_2gpu.txt (4 GiB
  // halves: 0.73 / 0.56 / 0.46 / 0.60 for 64 / 32 / 16 / 8-byte runs) scaled by 0.7, what the 16 GiB halves of the 33-qubit
  // run showed for 32-byte runs (268 GB/s per direction, profiles/r2_bench_2gpu_33q_tc_v2.json)
  double run_efficiency(int pos) const {
    const long run = (long)amp_bytes << pos;
    return run >= 128 ? 1.0 : run >= 64 ? 0.51 : run >= 32 ? 0.39 : run >= 16 ? 0.32 : 0.42;
  }
};

inline double plan_cost(const Plan& plan, const CostModel& m) {
  double ms = 0;
  const std::vector<Step>& st = plan.steps;
  for (size_t i = 0; i < st.size(); i++) {
    if (st[i].type == ST_TILE) ms += m.tile_ms;
    else if (st[i].type == ST_GATE) ms += m.gate_ms;
    else if (st[i].type == ST_SWAP) {
      // the run of swaps the executor would merge (Circuit::swap_run): distinct global bits and positions, at most 3
      int gb[3], lp[3], k = 0;
      size_t j = i;
      for (; j < st.size() && k < 3 && st[j].type == ST_SWAP; j++) {
        bool clash = false;
        for (int t = 0; t < k; t++) clash |= gb[t] == st[j].gbit || lp[t] == st[j].lpos;
        if (clash) break;
        gb[k] = st[j].gbit;
        lp[k] = st[j].lpos;
        k++;
      }
      bool can_merge = m.merged && k >= 2;
      for (int t = 0; t < k; t++) can_merge &= lp[t] >= m.vec_log2;
      if (!can_merge) k = 1;
      int low = lp[0];
      for (int t = 1; t < k; t++) low = lp[t] < low ? lp[t] : low;
      const double frac = k == 1 ? 0.5 : (1.0 - 1.0 / (1 << k)) / 0.91;   // merged: 0.91 of the single-swap rate (4 x B200)
      ms += 3.0 * frac * m.shard_ms / m.run_efficiency(low);            // state forward, state + adjoint in reverse
      i += (size_t)(k - 1);
    }
  }
  return ms;
}

// The plan of the cheapest candidate swap_min_pos in {opt.swap_min_pos, ..., 0} (ties: the highest position).
inline Plan schedule_best(const std::vector<SchedInst>& insts, const SchedOptions& opt, const CostModel& m, int* chosen_min_pos) {
  Plan best;
  double best_ms = -1;
  for (int mp = opt.swap_min_pos; mp >= 0; mp--) {
    SchedOptions o = opt;
    o.swap_min_pos = mp;
    Scheduler sch(insts, o);
    Plan p = sch.run();
    if (!p.ok) continue;
    const double ms = plan_cost(p, m);
    if (best_ms < 0 || ms < best_ms * (1.0 - 1e-9)) {
      best = p;
      best_ms = ms;
      if (chosen_min_pos) *chosen_min_pos = mp;
    }
  }
  if (best_ms < 0) {   // nothing schedulable: report the failure of the default options
    Scheduler sch(insts, opt);
    best = sch.run();
    if (chosen_min_pos) *chosen_min_pos = opt.swap_min_pos;
  }
  return best;
}

}  // namespace qdc
