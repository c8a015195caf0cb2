// Batched reduced density matrices and batched density seeds (SURVEY.md 8(f) item 2).
//
// The reference evaluates every requested density with its own sweep over the
// state and seeds every differentiable density with its own conj_and_double +
// gate + add sweeps (src/circuit.rs:252-257, 393-420; example_vqse_ising.py:77-79
// asks for n of them at one program point).  Here all densities of one program
// point whose qubits fit a tile are served by ONE sweep: a persistent CTA loads a
// tile of 2^T amplitudes into shared memory (same geometry / addressing as the
// gate passes) and
//   k_tile_dens : accumulates rho_d += psi (x) conj(psi) for every density d of the
//                 group (1*S bytes for the group instead of 1*S per density);
//   k_tile_seed : adds G_d^T (2 conj psi) for every differentiable density d into
//                 the adjoint tile (2*S or 3*S bytes for the group, not per density).
// Reductions follow the gradient reduction of k_tile_bwd: thread -> warp
// reduce-scatter -> CTA doubles kept across the CTA's tiles -> fixed-order final sum.
#pragma once
#include "tile_kernels.cuh"

#define QDC_TILE_MAXD 16
#define QDC_TILE_NT_D 128

struct TileDens {
  int type, a, b, slot;  // TG_Q1 (a) / TG_Q2 (a > b), tile-local positions; slot = result slot (k_tile_dens)
  GateMat tr;            // k_tile_seed: G^T in (hi,lo) order
};
struct TileDensParams {
  TileGeo geo;
  int ndens, live;       // live: the adjoint exists already (seed accumulates), else it is created
  TileDens d[QDC_TILE_MAXD];
};

template <int NT, class Geo>
__device__ __forceinline__ void tile_dens_items(const vec_t* smv, const Geo& geo, int nitems, real_t* acc) {
  constexpr int K = Geo::K;
  for (int i0 = 0; i0 < nitems; i0 += NT) {  // uniform trip count
    VecU v[Geo::NVEC];
    const uint32_t base = geo.base32((uint32_t)(i0 + threadIdx.x));
#pragma unroll
    for (int c = 0; c < Geo::NVEC; c++) v[c].v = smv[base + geo.off32(c)];
    cplx_t a[Geo::NG][K];
    Geo::unpack(v, a);
#pragma unroll
    for (int e = 0; e < Geo::NG; e++) dens_acc<K>(a[e], acc);
  }
}

// partials: [gridDim.x][ndens][32] doubles
__global__ void __launch_bounds__(QDC_TILE_NT_D, 3)
    k_tile_dens(const cplx_t* __restrict__ state, const __grid_constant__ TileDensParams p,
                double* __restrict__ partials) {
  extern __shared__ __align__(16) unsigned char tile_smem[];
  const int nvec = 1 << (p.geo.T - QDC_LV);
  vec_t* smv = (vec_t*)tile_smem;
  double* sm_acc = (double*)(smv + nvec);                      // [MAXD][32]
  real_t* sm_part = (real_t*)(sm_acc + QDC_TILE_MAXD * 32);      // [2][warps][32]
  constexpr int NW = QDC_TILE_NT_D / 32;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < QDC_TILE_MAXD * 32; i += QDC_TILE_NT_D) sm_acc[i] = 0.0;
  __syncthreads();
  TileAddr<QDC_TILE_NT_D> ta;
  ta.init(p.geo);
  for (uint64_t tile = blockIdx.x; tile < p.geo.ntiles; tile += gridDim.x) {
    tile_io<QDC_TILE_NT_D, true>((vec_t*)state, smv, ta, p.geo.tile(tile) >> QDC_LV);
    __syncthreads();
    for (int d = 0; d < p.ndens; d++) {
      const TileDens& D = p.d[d];
      real_t acc[32];
#pragma unroll
      for (int k = 0; k < 32; k++) acc[k] = 0;
      if (D.type == TG_Q2) {
#ifndef QDC_F64
        if (D.b == 0) {
          GeoQ2LH geo;
          geo.hv = D.a - 1;
          tile_dens_items<QDC_TILE_NT_D>(smv, geo, nvec / 2, acc);
        } else
#endif
        {
          GeoQ2HH geo;
          geo.lv = D.b - QDC_LV;
          geo.hv = D.a - QDC_LV;
          tile_dens_items<QDC_TILE_NT_D>(smv, geo, nvec / 4, acc);
        }
      } else {
#ifndef QDC_F64
        if (D.a == 0) {
          GeoQ1L geo;
          tile_dens_items<QDC_TILE_NT_D>(smv, geo, nvec, acc);
        } else
#endif
        {
          GeoQ1H geo;
          geo.pv = D.a - QDC_LV;
          tile_dens_items<QDC_TILE_NT_D>(smv, geo, nvec / 2, acc);
        }
      }
      real_t* part = sm_part + (size_t)(d & 1) * NW * 32;
      double s = 0.0;
      warp_flush<32>(acc, s, lane);
      part[warp * 32 + lane] = (real_t)s;
      __syncthreads();
      if (warp == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < NW; w++) t += (double)part[w * 32 + lane];
        sm_acc[d * 32 + lane] += t;
      }
    }
    __syncthreads();  // the tile and both halves of sm_part are free again
  }
  for (int i = threadIdx.x; i < p.ndens * 32; i += QDC_TILE_NT_D)
    partials[(size_t)blockIdx.x * p.ndens * 32 + i] = sm_acc[i];
}

template <int NT, class Geo>
__device__ __forceinline__ void tile_seed_items(const vec_t* smf, vec_t* smb, const Geo& geo, int nitems,
                                                const GateMat& G) {
  constexpr int K = Geo::K;
  for (int i0 = 0; i0 < nitems; i0 += NT) {  // uniform trip count
    VecU vf[Geo::NVEC], vb[Geo::NVEC];
    const uint32_t base = geo.base32((uint32_t)(i0 + threadIdx.x));
#pragma unroll
    for (int c = 0; c < Geo::NVEC; c++) {
      vf[c].v = smf[base + geo.off32(c)];
      vb[c].v = smb[base + geo.off32(c)];
    }
    cplx_t a[Geo::NG][K], b[Geo::NG][K];
    Geo::unpack(vf, a);
    Geo::unpack(vb, b);
#pragma unroll
    for (int e = 0; e < Geo::NG; e++) {
#pragma unroll
      for (int c = 0; c < K; c++) {  // t = 2 conj(psi)
        a[e][c].x = 2 * a[e][c].x;
        a[e][c].y = -2 * a[e][c].y;
      }
      mv<K>(G, a[e]);
#pragma unroll
      for (int c = 0; c < K; c++) {
        b[e][c].x += a[e][c].x;
        b[e][c].y += a[e][c].y;
      }
    }
    Geo::pack(vb, b);
#pragma unroll
    for (int c = 0; c < Geo::NVEC; c++) smb[base + geo.off32(c)] = vb[c].v;
  }
}

__global__ void __launch_bounds__(QDC_TILE_NT_D, 3)
    k_tile_seed(const cplx_t* __restrict__ fwd, cplx_t* __restrict__ bwd, const __grid_constant__ TileDensParams p) {
  extern __shared__ __align__(16) unsigned char tile_smem[];
  const int nvec = 1 << (p.geo.T - QDC_LV);
  vec_t* smf = (vec_t*)tile_smem;
  vec_t* smb = smf + nvec;
  TileAddr<QDC_TILE_NT_D> ta;
  ta.init(p.geo);
  for (uint64_t tile = blockIdx.x; tile < p.geo.ntiles; tile += gridDim.x) {
    const uint64_t tbase = p.geo.tile(tile) >> QDC_LV;
    tile_io<QDC_TILE_NT_D, true>((vec_t*)fwd, smf, ta, tbase);
    if (p.live) {
      tile_io<QDC_TILE_NT_D, true>((vec_t*)bwd, smb, ta, tbase);
    } else {
      VecU z;
#pragma unroll
      for (int k = 0; k < QDC_VR; k++) z.r[k] = 0;
      for (int i = threadIdx.x; i < nvec; i += QDC_TILE_NT_D) smb[i] = z.v;
    }
    __syncthreads();
    for (int d = 0; d < p.ndens; d++) {
      const TileDens& D = p.d[d];
      if (D.type == TG_Q2) {
#ifndef QDC_F64
        if (D.b == 0) {
          GeoQ2LH geo;
          geo.hv = D.a - 1;
          tile_seed_items<QDC_TILE_NT_D>(smf, smb, geo, nvec / 2, D.tr);
        } else
#endif
        {
          GeoQ2HH geo;
          geo.lv = D.b - QDC_LV;
          geo.hv = D.a - QDC_LV;
          tile_seed_items<QDC_TILE_NT_D>(smf, smb, geo, nvec / 4, D.tr);
        }
      } else {
#ifndef QDC_F64
        if (D.a == 0) {
          GeoQ1L geo;
          tile_seed_items<QDC_TILE_NT_D>(smf, smb, geo, nvec, D.tr);
        } else
#endif
        {
          GeoQ1H geo;
          geo.pv = D.a - QDC_LV;
          tile_seed_items<QDC_TILE_NT_D>(smf, smb, geo, nvec / 2, D.tr);
        }
      }
      __syncthreads();
    }
    tile_io<QDC_TILE_NT_D, false>((vec_t*)bwd, smb, ta, tbase);
    __syncthreads();
  }
}

// ------------------------------------------------------------ host side
// Greedy grouping of the densities of one program point: a group's positions (plus the
// forced low positions) must fit a tile of T positions and QDC_TILE_MAXD entries.
struct DensGroup {
  std::vector<int> steps;  // indices into plan_.steps
  std::vector<int> bits;   // physical positions of the tile
};

static inline std::vector<DensGroup> group_densities(const std::vector<qdc::Step>& steps, const std::vector<int>& which,
                                                     int T, int low_bits) {
  std::vector<DensGroup> out;
  DensGroup cur;
  auto fresh = [&]() {
    cur = DensGroup();
    for (int p = 0; p < low_bits; p++) cur.bits.push_back(p);
  };
  fresh();
  for (int si : which) {
    const qdc::Step& st = steps[si];
    int need = 0;
    if (std::find(cur.bits.begin(), cur.bits.end(), st.p2) == cur.bits.end()) need++;
    if (st.p1 >= 0 && std::find(cur.bits.begin(), cur.bits.end(), st.p1) == cur.bits.end()) need++;
    if (!cur.steps.empty() && ((int)cur.bits.size() + need > T || (int)cur.steps.size() == QDC_TILE_MAXD)) {
      out.push_back(cur);
      fresh();
    }
    if (std::find(cur.bits.begin(), cur.bits.end(), st.p2) == cur.bits.end()) cur.bits.push_back(st.p2);
    if (st.p1 >= 0 && std::find(cur.bits.begin(), cur.bits.end(), st.p1) == cur.bits.end()) cur.bits.push_back(st.p1);
    cur.steps.push_back(si);
  }
  if (!cur.steps.empty()) out.push_back(cur);
  return out;
}

inline const char* Circuit::fill_dens_params(const DensGroup& g, TileDensParams* p, std::vector<int>* tpos) {
  QDC_TRY(make_tile_geo_bits(g.bits, n_loc_, 0, &p->geo, tpos));
  p->ndens = (int)g.steps.size();
  for (int k = 0; k < p->ndens; k++) {
    const qdc::Step& st = plan_.steps[g.steps[k]];
    TileDens& D = p->d[k];
    if (st.p1 < 0) {
      D.type = TG_Q1;
      D.a = (*tpos)[st.p2];
      D.b = -1;
    } else {
      const bool swap = st.p2 < st.p1;
      D.type = TG_Q2;
      D.a = (*tpos)[swap ? st.p1 : st.p2];
      D.b = (*tpos)[swap ? st.p2 : st.p1];
    }
    D.slot = -1;
  }
  return nullptr;
}

// all densities of `g` in one sweep; results land in d_res_ slots (kernel (hi,lo) order, like eng_dens_q2)
inline const char* Circuit::run_dens_group(const DensGroup& g, const std::vector<long>& dslot) {
  static thread_local TileDensParams p;
  std::vector<int> tpos;
  QDC_TRY(fill_dens_params(g, &p, &tpos));
  p.live = 0;
  TileSlots h_slots;
  for (int k = 0; k < p.ndens; k++) h_slots.s[k] = p.d[k].slot = (int)dslot[plan_.steps[g.steps[k]].inst];
  const size_t smem = (sizeof(cplx_t) << p.geo.T) + QDC_TILE_MAXD * 32 * sizeof(double) +
                      2 * (QDC_TILE_NT_D / 32) * 32 * sizeof(real_t);
  int grid = 0;
  QDC_TRY(tile_grid((const void*)k_tile_dens, QDC_TILE_NT_D, smem, p.geo.ntiles, &grid));
  const size_t need = (size_t)grid * QDC_TILE_MAXG_B * 32;
  if (need > tile_partials_cap_) {
    if (tile_partials_) QDC_CUDA(cudaFree(tile_partials_));
    QDC_CUDA(cudaMalloc((void**)&tile_partials_, need * sizeof(double)));
    tile_partials_cap_ = need;
  }
  cudaEvent_t pa = nullptr;
  if (prof_.on) pa = prof_.begin(stream_);
  k_tile_dens<<<grid, QDC_TILE_NT_D, smem, stream_>>>(state_, p, tile_partials_);
  QDC_CUDA(cudaGetLastError());
  k_tile_final<<<p.ndens, 32, 0, stream_>>>(tile_partials_, grid, p.ndens, h_slots, d_res_);
  QDC_CUDA(cudaGetLastError());
  if (prof_.on) prof_.end(stream_, CAT_DENSITY, pa, (uint64_t)p.ndens * bytes());
  stats_.kernel_launches += 2;
  stats_.hbm_passes += 1;
  stats_.algorithmic_bytes += (uint64_t)p.ndens * bytes();
  return nullptr;
}

// bwd (+)= sum_d G_d^T (2 conj fwd) for the differentiable densities of `g` in one sweep
inline const char* Circuit::run_seed_group(const DensGroup& g, const std::vector<const cplx_t*>& dp, bool live) {
  static thread_local TileDensParams p;
  std::vector<int> tpos;
  QDC_TRY(fill_dens_params(g, &p, &tpos));
  p.live = live ? 1 : 0;
  for (int k = 0; k < p.ndens; k++) {
    const qdc::Step& st = plan_.steps[g.steps[k]];
    const bool swap = st.p1 >= 0 && st.p2 < st.p1;
    QDC_TRY(tile_matrix(dp[st.inst], st.p1 < 0 ? K_CONST_Q1 : K_CONST_Q2, FORM_TR, swap, &p.d[k].tr));
  }
  const size_t smem = 2 * (sizeof(cplx_t) << p.geo.T);
  int grid = 0;
  QDC_TRY(tile_grid((const void*)k_tile_seed, QDC_TILE_NT_D, smem, p.geo.ntiles, &grid));
  cudaEvent_t pa = nullptr;
  if (prof_.on) pa = prof_.begin(stream_);
  k_tile_seed<<<grid, QDC_TILE_NT_D, smem, stream_>>>(state_, bwd_, p);
  QDC_CUDA(cudaGetLastError());
  const uint64_t alg = (uint64_t)(live ? 3 : 2) + 3ull * (p.ndens - 1);  // per-density accounting of SURVEY 8(d)
  if (prof_.on) prof_.end(stream_, CAT_SEED, pa, alg * bytes());
  stats_.kernel_launches += 1;
  stats_.hbm_passes += 1;
  stats_.algorithmic_bytes += alg * bytes();
  return nullptr;
}

// The densities plan_.steps[first..last] belong to one program point: group them into tiled sweeps
// (singletons and the per-instruction executor keep the streaming kernels; k-qubit densities have sweeps of
// their own, dens_k_kernels.cuh).
inline const char* Circuit::run_dens_run(size_t first, size_t last, const std::vector<long>& dslot) {
  std::vector<int> which;
  for (size_t k = first; k <= last; k++) {
    if (plan_.steps[k].nk > 0) QDC_TRY(dens_k(plan_.steps[k]));
    else which.push_back((int)k);
  }
  const qdc::SchedOptions so = base_options();
  if (!opt_batch_dens_ || so.tile_bits == 0 || which.size() <= 1) {
    for (int k : which) QDC_TRY(dens_single(plan_.steps[k], dslot));
    return nullptr;
  }
  for (const DensGroup& g : group_densities(plan_.steps, which, so.tile_bits, so.low_bits)) {
    if (g.steps.size() == 1) QDC_TRY(dens_single(plan_.steps[g.steps[0]], dslot));
    else QDC_TRY(run_dens_group(g, dslot));
  }
  return nullptr;
}

inline const char* Circuit::run_seed_run(size_t first, size_t last, const std::vector<const cplx_t*>& dp, bool* live) {
  std::vector<int> which;  // differentiable densities only, in reverse program order like the reference
  for (size_t k = last + 1; k-- > first;) {
    if (!kind_is_diff_dens(insts_[plan_.steps[k].inst].kind)) continue;
    if (plan_.steps[k].nk > 0) {   // k-qubit densities: a seed sweep each
      QDC_TRY(seed_k(plan_.steps[k], *live));
      *live = true;
    } else {
      which.push_back((int)k);
    }
  }
  if (which.empty()) return nullptr;
  const qdc::SchedOptions so = base_options();
  if (!opt_batch_dens_ || so.tile_bits == 0 || which.size() == 1) {
    for (int k : which) {
      QDC_TRY(seed_single(plan_.steps[k], dp, *live));
      *live = true;
    }
    return nullptr;
  }
  for (const DensGroup& g : group_densities(plan_.steps, which, so.tile_bits, so.low_bits)) {
    if (g.steps.size() == 1) QDC_TRY(seed_single(plan_.steps[g.steps[0]], dp, *live));
    else QDC_TRY(run_seed_group(g, dp, *live));
    *live = true;
  }
  return nullptr;
}
