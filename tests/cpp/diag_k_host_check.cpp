// Host checks of the diagonal k-qubit gates (csrc/scheduler.hpp, csrc/diag_k_host.hpp), run by tests/test_diag_k.py:
//  * a sharded plan whose only instruction on global qubits is a diagonal k-qubit gate has no SWAP step, and the
//    gate is a wall: nothing is moved across it;
//  * the effective local diagonal of a gate with positions on rank bits (diag_fold) and the scatter of the kernel's
//    gradient to the gate's 2^k entries (diag_scatter) match a brute-force enumeration of the shard, for every rank
//    and every split of the positions between local and global.
#include <cmath>
#include <complex>
#include <cstdio>
#include <random>
#include <vector>

#include "diag_k_host.hpp"
#include "scheduler.hpp"

static int fails = 0;
#define CHECK(c)                                                   \
  do {                                                             \
    if (!(c)) {                                                    \
      if (fails++ < 20) printf("FAIL line %d: %s\n", __LINE__, #c); \
    }                                                              \
  } while (0)

static qdc::SchedInst q1(int q) { qdc::SchedInst s{}; s.kind_class = 0; s.q2 = q; s.q1 = -1; return s; }
static qdc::SchedInst q2(int a, int b) { qdc::SchedInst s{}; s.kind_class = 1; s.q2 = a; s.q1 = b; return s; }
static qdc::SchedInst kdiag(std::vector<int> qs) {
  qdc::SchedInst s{};
  s.kind_class = 7;
  s.q2 = s.q1 = -1;
  s.nq = (int)qs.size();
  for (size_t j = 0; j < qs.size(); j++) s.qk[j] = qs[j];
  return s;
}

static void check_plans() {
  for (int tile_bits : {0, 8}) {
    // n = 10 on 4 ranks (n_loc = 8): qubits 8 and 9 start global and only the diagonal touches them
    std::vector<qdc::SchedInst> in;
    for (int q = 0; q < 8; q++) in.push_back(q1(q));
    for (int q = 0; q + 1 < 8; q += 2) in.push_back(q2(q + 1, q));
    in.push_back(kdiag({9, 3, 8, 0}));
    in.push_back(q1(1));   // disjoint from the diagonal: must still run after it
    for (int q = 0; q < 8; q++) in.push_back(q1(q));
    in.push_back(kdiag({8, 9}));
    in.push_back(kdiag({9}));
    qdc::SchedOptions o;
    o.n = 10;
    o.n_loc = 8;
    o.tile_bits = tile_bits;
    o.low_bits = tile_bits ? 2 : 0;
    qdc::Scheduler sch(in, o);
    const qdc::Plan p = sch.run();
    CHECK(p.ok);
    int ndiag = 0, first_diag = -1, q1_after = -1;
    for (size_t i = 0; i < p.steps.size(); i++) {
      const qdc::Step& st = p.steps[i];
      CHECK(st.type != qdc::ST_SWAP);
      if (st.type == qdc::ST_DIAG_K) {
        CHECK(qdc::is_wall(st));
        if (first_diag < 0) first_diag = (int)i;
        ndiag++;
        CHECK(st.nk == in[st.inst].nq);
        for (int j = 0; j < st.nk; j++) CHECK(st.pk[j] == in[st.inst].qk[j]);   // no remap: identity positions
      }
      auto is_q1_after = [&](const qdc::Step& s) { return s.inst == 13; };
      if (st.type == qdc::ST_GATE && is_q1_after(st)) q1_after = (int)i;
      if (st.type == qdc::ST_TILE)
        for (int k = 0; k < st.count; k++)
          if (is_q1_after(p.tile_steps[st.first + k])) q1_after = (int)i;
    }
    CHECK(ndiag == 3);
    CHECK(first_diag >= 0 && q1_after > first_diag);
    for (int q = 0; q < 10; q++) CHECK(p.final_map[q] == q);
  }
}

static void check_fold() {
  std::mt19937 rng(7);
  std::normal_distribution<double> nd;
  const int n = 8;
  for (int k = 1; k <= 6; k++) {
    for (int trial = 0; trial < 6; trial++) {
      // k distinct positions in random order
      std::vector<int> perm(n);
      for (int i = 0; i < n; i++) perm[i] = i;
      std::shuffle(perm.begin(), perm.end(), rng);
      int pk[6];
      for (int q = 0; q < k; q++) pk[q] = perm[q];
      std::vector<std::complex<double>> d((size_t)1 << k);
      for (auto& v : d) v = {nd(rng), nd(rng)};
      for (int n_loc = 1; n_loc <= n; n_loc++) {   // every split of the positions between local and rank bits
        for (int rank = 0; rank < (1 << (n - n_loc)); rank++) {
          const qdc::DiagFold f = qdc::diag_fold_split(pk, k, n_loc, rank);
          std::vector<std::complex<double>> dl;
          qdc::diag_fold(f, k, d.data(), &dl);
          CHECK((int)dl.size() == (1 << f.k_loc));
          std::vector<double> gl((size_t)2 << f.k_loc, 0.0);
          std::vector<std::complex<double>> gfull((size_t)1 << k, 0.0);
          for (int il = 0; il < (1 << n_loc); il++) {
            const int i = il | (rank << n_loc);   // global amplitude index
            int j = 0, jl = 0;
            for (int q = 0; q < k; q++) j = (j << 1) | ((i >> pk[q]) & 1);
            for (int q = 0; q < f.k_loc; q++) jl = (jl << 1) | ((il >> f.loc[q]) & 1);
            CHECK(dl[jl] == d[j]);   // the effective local diagonal multiplies every amplitude by d[j]
            const double x = nd(rng), y = nd(rng);   // a contribution of this amplitude to the gradient
            gl[2 * jl] += x;
            gl[2 * jl + 1] += y;
            gfull[j] += std::complex<double>(x, y);
          }
          std::vector<std::complex<double>> g;
          qdc::diag_scatter(f, k, gl.data(), &g);
          CHECK(g.size() == gfull.size());
          for (size_t j = 0; j < g.size(); j++) CHECK(std::abs(g[j] - gfull[j]) < 1e-12);
        }
      }
    }
  }
}

int main() {
  check_plans();
  check_fold();
  if (fails) {
    printf("%d failures\n", fails);
    return 1;
  }
  printf("OK\n");
  return 0;
}
