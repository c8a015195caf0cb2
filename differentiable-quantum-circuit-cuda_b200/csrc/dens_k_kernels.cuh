// k-qubit reduced density matrices (3 <= k <= 6) and their backward seeds (kinds DENS_K / DIFF_DENS_K).
//
//   k_dens_k : rho[r, c] = sum_rest psi[r, rest] conj psi[c, rest]          (1*S bytes)
//   k_seed_k : bwd[r, rest] (+)= sum_c G[c, r] 2 conj fwd[c, rest]           (2*S created, 3*S accumulated)
// with r, c the k-bit index over `positions` (positions[0] is the most significant bit) and G the cotangent of the
// density, so the seed is (G^T acting on positions)(2 conj fwd), the k-qubit form of the one- and two-qubit seeds.
//
// A persistent CTA walks tiles of 2^T amplitudes whose positions are the k density positions, the low positions
// (coalesced runs) and padding: the same TileGeo / TileAddr / tile_io as the gate passes, so loads stay coalesced
// for any position set.  A single-tile register (n_loc <= T_max) is loaded as it is.  Inside the tile the amplitudes
// are re-staged as a D x (rest + 1) matrix (D = 2^k; the odd leading dimension keeps a warp's column reads on
// distinct banks), and each thread owns a 4 x 4 block of outputs:
//   density: the rows rb + Q i and columns cb + Q l (Q = D / 4) of rho, summed over a 1/S share of the rest index
//            (S = 256 / Q^2 threads per block); real_t per tile, double across the CTA's tiles, then a fixed-order
//            sum over (CTA, share) in k_dens_k_final -- no floating-point atomics, the same result run to run;
//   seed:    the rows rb + Q i and four rest columns of the new adjoint tile, written to the tile once.
// Cost (k = 6): 64 complex MACs per amplitude on the FP32 / FP64 pipe, against one read of the state.
#pragma once
#include "tile_kernels.cuh"

#define QDC_DENSK_NT 256
#define QDC_DENSK_MAXK 6

struct DensKParams {
  TileGeo geo;   // geo.T is the tile size in both modes
  int whole;     // 1: the whole register is one tile, in its own order (geo.hi / geo.tile unused)
  int live;      // seed: the adjoint exists already (accumulate), else it is created
  int a[QDC_DENSK_MAXK];  // tile-local bit of positions[j]
};

// roff[r]: tile offset of the density index r;  resto[j]: tile offset of the rest index j (the other tile bits,
// ascending)
template <int KQ>
__device__ __forceinline__ void dens_k_tables(const DensKParams& p, int* roff, int* resto) {
  constexpr int D = 1 << KQ;
  const int T = p.geo.T, nrest = 1 << (T - KQ);
  int mask = 0;
#pragma unroll
  for (int j = 0; j < KQ; j++) mask |= 1 << p.a[j];
  for (int r = threadIdx.x; r < D; r += QDC_DENSK_NT) {
    int off = 0;
#pragma unroll
    for (int j = 0; j < KQ; j++) off |= ((r >> (KQ - 1 - j)) & 1) << p.a[j];
    roff[r] = off;
  }
  for (int j = threadIdx.x; j < nrest; j += QDC_DENSK_NT) {
    int off = 0, b = 0;
    for (int t = 0; t < T; t++)
      if (!((mask >> t) & 1)) off |= ((j >> b++) & 1) << t;
    resto[j] = off;
  }
}

__device__ __forceinline__ void dens_k_load(const DensKParams& p, const TileAddr<QDC_DENSK_NT>& ta, cplx_t* gmem,
                                            cplx_t* sm, uint64_t tile) {
  if (p.whole) {
    for (int i = threadIdx.x; i < (1 << p.geo.T); i += QDC_DENSK_NT) sm[i] = gmem[i];
  } else {
    tile_io<QDC_DENSK_NT, true>((vec_t*)gmem, (vec_t*)sm, ta, p.geo.tile(tile) >> QDC_LV);
  }
}

// Y[r * ld + j] = scale * (conj) X[roff[r] | resto[j]]
template <int KQ, bool CONJ2>
__device__ __forceinline__ void dens_k_stage(const cplx_t* X, cplx_t* Y, const int* roff, const int* resto, int T,
                                             int ld) {
  const int rbits = T - KQ;
  for (int e = threadIdx.x; e < (1 << T); e += QDC_DENSK_NT) {
    const int r = e >> rbits, j = e & ((1 << rbits) - 1);
    cplx_t v = X[roff[r] | resto[j]];
    if (CONJ2) {
      v.x = 2 * v.x;
      v.y = -2 * v.y;
    }
    Y[r * ld + j] = v;
  }
}

template <int KQ>
__device__ __forceinline__ void dens_k_items(const cplx_t* Y, int ld, int nrest, int s, int rb, int cb,
                                             real_t (&acc)[32]) {
  constexpr int Q = (1 << KQ) / 4, S = QDC_DENSK_NT / (Q * Q);
  for (int j = s; j < nrest; j += S) {
    cplx_t a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      a[i] = Y[(rb + Q * i) * ld + j];
      b[i] = Y[(cb + Q * i) * ld + j];
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
#pragma unroll
      for (int l = 0; l < 4; l++) {  // a conj(b)
        acc[2 * (4 * i + l)] += a[i].x * b[l].x + a[i].y * b[l].y;
        acc[2 * (4 * i + l) + 1] += a[i].y * b[l].x - a[i].x * b[l].y;
      }
    }
  }
}

// partials: [gridDim.x][QDC_DENSK_NT][32] doubles (thread = share s * Q^2 + owner)
template <int KQ>
__global__ void __launch_bounds__(QDC_DENSK_NT, 1)
    k_dens_k(const cplx_t* __restrict__ state, const __grid_constant__ DensKParams p, double* __restrict__ partials) {
  constexpr int D = 1 << KQ, Q = D / 4, OWN = Q * Q;
  extern __shared__ __align__(16) unsigned char densk_smem[];
  const int T = p.geo.T, nrest = 1 << (T - KQ), ld = nrest + 1;
  cplx_t* X = (cplx_t*)densk_smem;
  cplx_t* Y = X + (1 << T);
  int* roff = (int*)(Y + D * ld);
  int* resto = roff + D;
  dens_k_tables<KQ>(p, roff, resto);
  TileAddr<QDC_DENSK_NT> ta;
  if (!p.whole) ta.init(p.geo);
  const int o = threadIdx.x % OWN, s = threadIdx.x / OWN, rb = o / Q, cb = o % Q;
  double dacc[32];
#pragma unroll
  for (int q = 0; q < 32; q++) dacc[q] = 0.0;
  const uint64_t ntiles = p.whole ? 1 : p.geo.ntiles;
  for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    dens_k_load(p, ta, (cplx_t*)state, X, tile);
    __syncthreads();
    dens_k_stage<KQ, false>(X, Y, roff, resto, T, ld);
    __syncthreads();
#ifdef QDC_F64
    dens_k_items<KQ>(Y, ld, nrest, s, rb, cb, dacc);
#else
    real_t acc[32];
#pragma unroll
    for (int q = 0; q < 32; q++) acc[q] = 0;
    dens_k_items<KQ>(Y, ld, nrest, s, rb, cb, acc);
#pragma unroll
    for (int q = 0; q < 32; q++) dacc[q] += (double)acc[q];
#endif
    __syncthreads();  // X and Y are free again
  }
  double* dst = partials + ((size_t)blockIdx.x * QDC_DENSK_NT + threadIdx.x) * 32;
#pragma unroll
  for (int q = 0; q < 32; q++) dst[q] = dacc[q];
}

// out[2 (r D + c) + re/im] = sum over (CTA, share) pairs, in order, of the owner's partials (one block per owner)
template <int KQ>
__global__ void __launch_bounds__(256)
    k_dens_k_final(const double* __restrict__ partials, int npairs, double* __restrict__ out) {
  constexpr int D = 1 << KQ, Q = D / 4, OWN = Q * Q;
  __shared__ double red[8][32];
  const int o = blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double s = 0.0;
  for (int pr = w; pr < npairs; pr += 8) s += partials[((size_t)pr * OWN + o) * 32 + lane];
  red[w][lane] = s;
  __syncthreads();
  if (w == 0) {
    double t = 0.0;
#pragma unroll
    for (int v = 0; v < 8; v++) t += red[v][lane];
    const int e = lane >> 1, i = e >> 2, l = e & 3;
    const int r = o / Q + Q * i, c = o % Q + Q * l;
    out[2 * (r * D + c) + (lane & 1)] = t;
  }
}

// bwd (+)= (G^T on the positions) (2 conj fwd);  G: D x D cotangent, row-major, in global memory
template <int KQ>
__global__ void __launch_bounds__(QDC_DENSK_NT, 1)
    k_seed_k(const cplx_t* __restrict__ fwd, cplx_t* __restrict__ bwd, const cplx_t* __restrict__ G,
             const __grid_constant__ DensKParams p) {
  constexpr int D = 1 << KQ, Q = D / 4;
  extern __shared__ __align__(16) unsigned char densk_smem[];
  const int T = p.geo.T, nrest = 1 << (T - KQ), ld = nrest + 1;
  cplx_t* X = (cplx_t*)densk_smem;
  cplx_t* Y = X + (1 << T);
  cplx_t* Gs = Y + D * ld;
  int* roff = (int*)(Gs + D * D);
  int* resto = roff + D;
  dens_k_tables<KQ>(p, roff, resto);
  for (int i = threadIdx.x; i < D * D; i += QDC_DENSK_NT) Gs[i] = G[i];
  TileAddr<QDC_DENSK_NT> ta;
  if (!p.whole) ta.init(p.geo);
  // items: (row block rb, rest columns jb + js l), consecutive threads on consecutive jb (G reads broadcast)
  const int nj = nrest >= 4 ? nrest / 4 : 1, js = nj, nitems = Q * nj;
  const uint64_t ntiles = p.whole ? 1 : p.geo.ntiles;
  for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    dens_k_load(p, ta, (cplx_t*)fwd, X, tile);
    __syncthreads();
    dens_k_stage<KQ, true>(X, Y, roff, resto, T, ld);
    __syncthreads();
    if (p.live) {
      dens_k_load(p, ta, bwd, X, tile);
      __syncthreads();
    }
    for (int it = threadIdx.x; it < nitems; it += QDC_DENSK_NT) {
      const int rb = it / nj, jb = it % nj;
      cplx_t acc[4][4];
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int l = 0; l < 4; l++) acc[i][l].x = acc[i][l].y = 0;
      for (int c = 0; c < D; c++) {
        cplx_t y[4], g[4];
#pragma unroll
        for (int l = 0; l < 4; l++) {
          const int j = jb + js * l;
          if (j < nrest) y[l] = Y[c * ld + j];
          else y[l].x = y[l].y = 0;
        }
#pragma unroll
        for (int i = 0; i < 4; i++) g[i] = Gs[c * D + rb + Q * i];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int l = 0; l < 4; l++) {
            acc[i][l].x += g[i].x * y[l].x - g[i].y * y[l].y;
            acc[i][l].y += g[i].x * y[l].y + g[i].y * y[l].x;
          }
      }
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int l = 0; l < 4; l++) {
          const int j = jb + js * l;
          if (j >= nrest) continue;
          cplx_t& dst = X[roff[rb + Q * i] | resto[j]];   // written by this thread only
          cplx_t v = acc[i][l];
          if (p.live) {
            v.x += dst.x;
            v.y += dst.y;
          }
          dst = v;
        }
    }
    __syncthreads();
    if (p.whole) {
      for (int i = threadIdx.x; i < (1 << T); i += QDC_DENSK_NT) bwd[i] = X[i];
    } else {
      tile_io<QDC_DENSK_NT, false>((vec_t*)bwd, (vec_t*)X, ta, p.geo.tile(tile) >> QDC_LV);
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------ host side
inline const char* Circuit::fill_dens_k_params(const qdc::Step& st, DensKParams* p) {
  memset(p, 0, sizeof(*p));
  std::vector<int> tpos;
  if (n_loc_ <= QDC_LV + 11) {   // the register fits one tile: load it as it is
    p->whole = 1;
    p->geo.T = n_loc_;
    p->geo.ntiles = 1;
    tpos.resize(n_loc_);
    for (int b = 0; b < n_loc_; b++) tpos[b] = b;
  } else {
    std::vector<int> bits;
    for (int b = 0; b < default_low_bits(); b++) bits.push_back(b);
    for (int j = 0; j < st.nk; j++)
      if (std::find(bits.begin(), bits.end(), st.pk[j]) == bits.end()) bits.push_back(st.pk[j]);
    QDC_TRY(make_tile_geo_bits(bits, n_loc_, 0, &p->geo, &tpos));
  }
  for (int j = 0; j < st.nk; j++) p->a[j] = tpos[st.pk[j]];
  return nullptr;
}

template <int KQ>
static inline size_t dens_k_smem(int T, bool seed) {
  constexpr int D = 1 << KQ;
  const int nrest = 1 << (T - KQ);
  return (sizeof(cplx_t) << T) + sizeof(cplx_t) * D * (nrest + 1) + (seed ? sizeof(cplx_t) * D * D : 0) +
         sizeof(int) * (D + nrest);
}

template <int KQ>
inline const char* Circuit::launch_dens_k(const DensKParams& p, double* dst) {
  constexpr int OWN = (1 << KQ) / 4 * ((1 << KQ) / 4), S = QDC_DENSK_NT / OWN;
  const size_t smem = dens_k_smem<KQ>(p.geo.T, false);
  int grid = 0;
  QDC_TRY(tile_grid((const void*)k_dens_k<KQ>, QDC_DENSK_NT, smem, p.whole ? 1 : p.geo.ntiles, &grid));
  const size_t need = (size_t)grid * QDC_DENSK_NT * 32;
  if (need > tile_partials_cap_) {
    if (tile_partials_) QDC_CUDA(cudaFree(tile_partials_));
    QDC_CUDA(cudaMalloc((void**)&tile_partials_, need * sizeof(double)));
    tile_partials_cap_ = need;
  }
  k_dens_k<KQ><<<grid, QDC_DENSK_NT, smem, stream_>>>(state_, p, tile_partials_);
  QDC_CUDA(cudaGetLastError());
  k_dens_k_final<KQ><<<OWN, 256, 0, stream_>>>(tile_partials_, grid * S, dst);
  QDC_CUDA(cudaGetLastError());
  return nullptr;
}

template <int KQ>
inline const char* Circuit::launch_seed_k(const DensKParams& p, const cplx_t* G) {
  const size_t smem = dens_k_smem<KQ>(p.geo.T, true);
  int grid = 0;
  QDC_TRY(tile_grid((const void*)k_seed_k<KQ>, QDC_DENSK_NT, smem, p.whole ? 1 : p.geo.ntiles, &grid));
  k_seed_k<KQ><<<grid, QDC_DENSK_NT, smem, stream_>>>(state_, bwd_, G, p);
  QDC_CUDA(cudaGetLastError());
  return nullptr;
}

inline const char* Circuit::dens_k(const qdc::Step& st) {
  static thread_local DensKParams p;
  QDC_TRY(fill_dens_k_params(st, &p));
  double* dst = d_kres_ + kofs_[st.inst];
  switch (st.nk) {
    case 3: PROF(CAT_DENSITY, 1, launch_dens_k<3>(p, dst)); break;
    case 4: PROF(CAT_DENSITY, 1, launch_dens_k<4>(p, dst)); break;
    case 5: PROF(CAT_DENSITY, 1, launch_dens_k<5>(p, dst)); break;
    case 6: PROF(CAT_DENSITY, 1, launch_dens_k<6>(p, dst)); break;
    default: return qdc_errf("internal: %d-qubit density step.", st.nk);
  }
  account(2, 1, 1);
  return nullptr;
}

inline const char* Circuit::seed_k(const qdc::Step& st, bool live) {
  static thread_local DensKParams p;
  QDC_TRY(fill_dens_k_params(st, &p));
  p.live = live ? 1 : 0;
  const cplx_t* G = d_kmat_ + kmat_ofs_[st.inst];
  switch (st.nk) {
    case 3: PROF(CAT_SEED, live ? 3 : 2, launch_seed_k<3>(p, G)); break;
    case 4: PROF(CAT_SEED, live ? 3 : 2, launch_seed_k<4>(p, G)); break;
    case 5: PROF(CAT_SEED, live ? 3 : 2, launch_seed_k<5>(p, G)); break;
    case 6: PROF(CAT_SEED, live ? 3 : 2, launch_seed_k<6>(p, G)); break;
    default: return qdc_errf("internal: %d-qubit density seed.", st.nk);
  }
  account(1, 1, live ? 3 : 2);
  return nullptr;
}
