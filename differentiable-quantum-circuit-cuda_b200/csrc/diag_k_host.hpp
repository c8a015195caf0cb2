// Host-only mathematics of the diagonal k-qubit gates on a sharded register (pure C++, no CUDA; compiled by the CPU
// test tests/cpp/diag_k_host_check.cpp as well).
//
// A diagonal gate d on physical positions pk[0..k-1] (pk[0] the most significant bit of j) needs no exchange: on the
// rank `rank` every position >= n_loc is a rank bit with a fixed value, so the gate acts on the shard as the diagonal
//   d_loc[j_loc] = d[j(j_loc, the rank's bits)]
// over the k_loc local positions (in the same relative order).  k_loc = 0 is a scalar multiply of the shard.  The
// kernel's 2^k_loc gradient entries G_loc are the entries of the full 2^k gradient whose global bits equal the rank's;
// the other entries are zero on this rank (the ranks' partial gradients are summed by the caller's all-reduce).
#pragma once
#include <complex>
#include <vector>

namespace qdc {

struct DiagFold {
  int k_loc = 0;
  int loc[6] = {-1, -1, -1, -1, -1, -1};   // the local physical positions, most significant first
  int gmask = 0, gval = 0;                  // bits of j on rank positions, and their value on this rank
};

// Split the positions of a k-qubit diagonal into local positions and rank bits.
inline DiagFold diag_fold_split(const int* pk, int k, int n_loc, int rank) {
  DiagFold f;
  for (int q = 0; q < k; q++) {
    const int bit = 1 << (k - 1 - q);
    if (pk[q] >= n_loc) {
      f.gmask |= bit;
      if ((rank >> (pk[q] - n_loc)) & 1) f.gval |= bit;
    } else {
      f.loc[f.k_loc++] = pk[q];
    }
  }
  return f;
}

// j of the full gate from the local index j_loc (k_loc bits, most significant first) and the rank's bits
inline int diag_fold_index(const DiagFold& f, int k, int j_loc) {
  int j = f.gval, b = f.k_loc;
  for (int q = 0; q < k; q++) {
    const int bit = 1 << (k - 1 - q);
    if (f.gmask & bit) continue;
    b--;
    if ((j_loc >> b) & 1) j |= bit;
  }
  return j;
}

// d_loc[j_loc] = d[diag_fold_index(j_loc)], 2^k_loc entries
template <class C>
inline void diag_fold(const DiagFold& f, int k, const C* d, std::vector<C>* out) {
  out->resize((size_t)1 << f.k_loc);
  for (int jl = 0; jl < (1 << f.k_loc); jl++) (*out)[jl] = d[diag_fold_index(f, k, jl)];
}

// The full 2^k gradient on this rank from the kernel's 2^k_loc entries (interleaved re / im doubles): zero where the
// rank bits of j differ from the rank's.
inline void diag_scatter(const DiagFold& f, int k, const double* g_loc, std::vector<std::complex<double>>* out) {
  out->assign((size_t)1 << k, std::complex<double>(0, 0));
  for (int jl = 0; jl < (1 << f.k_loc); jl++)
    (*out)[diag_fold_index(f, k, jl)] = std::complex<double>(g_loc[2 * jl], g_loc[2 * jl + 1]);
}

}  // namespace qdc
