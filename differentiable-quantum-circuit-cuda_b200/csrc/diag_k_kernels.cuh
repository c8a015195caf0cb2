// Diagonal gates on k = 1..6 qubits and their reverse steps (kinds CONST_DIAG_K / VAR_DIAG_K / *_NONU).
//
//   k_diag_k     : psi[j, rest] = d[j] psi[j, rest]                                            (2*S, in place)
//   k_diag_k_rev : fwd <- a fwd;  G[j] = sum_rest bwd[j, rest] fwd[j, rest];  bwd <- d bwd          (4*S)
// with j the k-bit index over `positions` (positions[0] is the most significant bit).  k_diag_k applies d in the
// forward pass and the un-compute form a (conj d, or 1 / d for NonU gates) in the reverse pass while no adjoint exists;
// k_diag_k_rev is the reverse step of the two-qubit diagonal (EOpDiagRev) at width k: the gradient without
// conjugation from the un-computed state and the adjoint before the pull-back, and U^T = U.
//
// Both are single elementwise sweeps with 128-bit accesses and several loads in flight per thread.  The entries are
// staged in shared memory (a per-amplitude select from kernel parameters is a divergent constant-bank access: 4x
// slower, DESIGN.md 4 "Diagonal gates").
//   * k_diag_k streams the register linearly (every access coalesced, whatever the positions).
//   * k_diag_k_rev walks the tiles of the k-qubit densities (fill_dens_k_params: the k positions and the low bits
//     inside a tile of 2^T amplitudes, TileAddr / tile runs of >= 128 bytes) straight from HBM into registers; no tile
//     is staged.  Every thread owns the same S = NI * QDC_VA in-tile amplitudes in every tile, so each of its S
//     gradient accumulators always belongs to the same j.  They are summed in real_t over QDC_DIAGK_FLUSH tiles, then
//     added into the thread's doubles in shared memory; at the end the CTA sums its (thread, slot) doubles into the 2^k
//     bins in a fixed order, and k_diag_k_final sums the CTAs in a fixed order: no floating-point atomics, the same
//     result run to run.
// A register that fits one tile (n_loc <= QDC_LV + 11) runs the reverse step in one CTA (k_diag_k_rev_whole).
// On a sharded register the positions on rank bits are folded into the entries on the host (diag_k_host.hpp), so
// the kernels see k_loc <= k local positions; k_loc = 0 is a scalar multiply.
#pragma once
#include "dens_k_kernels.cuh"

#define QDC_DIAGK_NT 256      // threads of the reverse step (the k-density tile walk: TileAddr<256>)
#define QDC_DIAGK_FLUSH 8     // tiles between flushes of the real_t gradient accumulators into doubles
#define QDC_DIAGK_UNROLL 4    // vectors in flight per thread in k_diag_k

struct DiagKPos {
  int nk;       // local positions of the gate (0..6)
  int pos[6];   // their bits in the amplitude index (physical, or tile-local for the reverse step), most significant
                // first
};

// (unrolled over the 6 slots: a run-time index into a kernel parameter array would copy it to the stack)
__device__ __forceinline__ int diag_k_index(uint64_t amp, const DiagKPos& p) {
  int j = 0;
#pragma unroll
  for (int q = 0; q < 6; q++)
    if (q < p.nk) j = (j << 1) | (int)((amp >> p.pos[q]) & 1ull);
  return j;
}

// (re, im) <- d (re, im)
__device__ __forceinline__ void diag_k_mul(const cplx_t d, real_t& re, real_t& im) {
  const real_t r = d.x * re - d.y * im;
  im = d.x * im + d.y * re;
  re = r;
}

// buf[j, rest] *= d[j]
__global__ void __launch_bounds__(QDC_BLOCK)
    k_diag_k(vec_t* __restrict__ buf, const cplx_t* __restrict__ d, const DiagKPos p, const uint64_t nvec) {
  constexpr int U = QDC_DIAGK_UNROLL;
  __shared__ cplx_t ds[64];
  for (int i = threadIdx.x; i < (1 << p.nk); i += QDC_BLOCK) ds[i] = d[i];
  __syncthreads();
  const uint64_t stride = (uint64_t)gridDim.x * QDC_BLOCK;
  for (uint64_t v0 = (uint64_t)blockIdx.x * QDC_BLOCK + threadIdx.x; v0 < nvec; v0 += stride * U) {
    VecU x[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t v = v0 + (uint64_t)u * stride;
      if (v < nvec) x[u].v = buf[v];
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t v = v0 + (uint64_t)u * stride;
      if (v < nvec) {
#pragma unroll
        for (int e = 0; e < QDC_VA; e++)
          diag_k_mul(ds[diag_k_index((v << QDC_LV) | (uint64_t)e, p)], x[u].r[2 * e], x[u].r[2 * e + 1]);
        buf[v] = x[u].v;
      }
    }
  }
}

// The tile-local amplitude index with j = b and rest index r (rest = the tile bits that are not positions, ascending)
__device__ __forceinline__ int diag_k_deposit(int b, int r, const DiagKPos& p, int T) {
  int e = 0, mask = 0;
#pragma unroll
  for (int q = 0; q < 6; q++) {
    if (q >= p.nk) continue;
    mask |= 1 << p.pos[q];
    e |= ((b >> (p.nk - 1 - q)) & 1) << p.pos[q];
  }
  for (int t = 0, bit = 0; t < T; t++)
    if (!((mask >> t) & 1)) e |= ((r >> bit++) & 1) << t;
  return e;
}

// out[b] (interleaved re / im) = sum over the CTAs, in order, of partials[cta][b] (one block per bin)
__global__ void __launch_bounds__(256)
    k_diag_k_final(const double2* __restrict__ partials, int ncta, double* __restrict__ out) {
  __shared__ double2 red[256];
  const int b = blockIdx.x;
  double2 s = make_double2(0.0, 0.0);
  for (int c = threadIdx.x; c < ncta; c += 256) {
    const double2 v = partials[(size_t)c * 64 + b];
    s.x += v.x;
    s.y += v.y;
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int h = 128; h > 0; h >>= 1) {
    if (threadIdx.x < h) {
      red[threadIdx.x].x += red[threadIdx.x + h].x;
      red[threadIdx.x].y += red[threadIdx.x + h].y;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[2 * b] = red[0].x;
    out[2 * b + 1] = red[0].y;
  }
}

// Reverse step over the tiles of p (p.pos: tile-local bits).  A: the un-compute form, B: d, both 2^nk entries.
// partials (variable gates; nullptr for constant ones): [gridDim.x][64] double2, summed by k_diag_k_final.
// Dynamic shared memory (variable gates): S * QDC_DIAGK_NT double2, the threads' gradient accumulators.
template <int NI>
__global__ void __launch_bounds__(QDC_DIAGK_NT, 2)
    k_diag_k_rev(vec_t* __restrict__ fwd, vec_t* __restrict__ bwd, const cplx_t* __restrict__ A,
                 const cplx_t* __restrict__ B, const __grid_constant__ TileGeo geo, const DiagKPos p,
                 double2* __restrict__ partials) {
  constexpr int NT = QDC_DIAGK_NT, S = NI * QDC_VA, NH = NI < 4 ? NI : 4;
  extern __shared__ __align__(16) unsigned char diagk_smem[];
  __shared__ cplx_t As[64], Bs[64];
  __shared__ double2 shares[NT];
  double2* red = (double2*)diagk_smem;   // [slot][thread]
  const int tid = threadIdx.x;
  const bool grad = partials != nullptr;
  for (int i = tid; i < (1 << p.nk); i += NT) {
    As[i] = A[i];
    Bs[i] = B[i];
  }
  if (grad)
    for (int s = 0; s < S; s++) red[s * NT + tid] = make_double2(0.0, 0.0);
  TileAddr<NT> ta;
  ta.init(geo);
  int js[S];   // j of every slot: the same in every tile
#pragma unroll
  for (int s = 0; s < S; s++) js[s] = diag_k_index((uint64_t)(((tid + (s / QDC_VA) * NT) << QDC_LV) | (s % QDC_VA)), p);
  real_t acc[2 * S];
#pragma unroll
  for (int q = 0; q < 2 * S; q++) acc[q] = 0;
  __syncthreads();
  int since = 0;
  for (uint64_t tile = blockIdx.x; tile < geo.ntiles; tile += gridDim.x) {
    const uint64_t base = (geo.tile(tile) >> QDC_LV) + ta.lo;
#pragma unroll
    for (int h = 0; h < NI; h += NH) {   // NH vectors of state and adjoint in flight
      VecU f[NH], b[NH];
#pragma unroll
      for (int i = 0; i < NH; i++) {
        const uint64_t v = base + ((uint64_t)ta.it[h + i] << ta.runv_log);
        f[i].v = fwd[v];
        b[i].v = bwd[v];
      }
#pragma unroll
      for (int i = 0; i < NH; i++) {
#pragma unroll
        for (int e = 0; e < QDC_VA; e++) {
          const int s = (h + i) * QDC_VA + e;
          real_t &fr = f[i].r[2 * e], &fi = f[i].r[2 * e + 1], &br = b[i].r[2 * e], &bi = b[i].r[2 * e + 1];
          diag_k_mul(As[js[s]], fr, fi);
          if (grad) {   // bwd fwd, no conjugation
            acc[2 * s] += br * fr - bi * fi;
            acc[2 * s + 1] += br * fi + bi * fr;
          }
          diag_k_mul(Bs[js[s]], br, bi);
        }
      }
#pragma unroll
      for (int i = 0; i < NH; i++) {
        const uint64_t v = base + ((uint64_t)ta.it[h + i] << ta.runv_log);
        fwd[v] = f[i].v;
        bwd[v] = b[i].v;
      }
    }
    if (grad && ++since == QDC_DIAGK_FLUSH) {
#pragma unroll
      for (int s = 0; s < S; s++) {
        red[s * NT + tid].x += (double)acc[2 * s];
        red[s * NT + tid].y += (double)acc[2 * s + 1];
        acc[2 * s] = acc[2 * s + 1] = 0;
      }
      since = 0;
    }
  }
  if (!grad) return;
#pragma unroll
  for (int s = 0; s < S; s++) {
    red[s * NT + tid].x += (double)acc[2 * s];
    red[s * NT + tid].y += (double)acc[2 * s + 1];
  }
  __syncthreads();
  // bins: G threads per j, each summing a fixed share of the rest index; then the shares in order
  const int D = 1 << p.nk, G = NT / D, bin = tid / G, g = tid % G, nrest = 1 << (geo.T - p.nk);
  double2 sum = make_double2(0.0, 0.0);
  for (int r = g; r < nrest; r += G) {
    const int e = diag_k_deposit(bin, r, p, geo.T);
    const double2 v = red[((e & (QDC_VA - 1)) + ((e >> (QDC_LV + 8)) * QDC_VA)) * NT + ((e >> QDC_LV) & (NT - 1))];
    sum.x += v.x;
    sum.y += v.y;
  }
  shares[tid] = sum;
  __syncthreads();
  if (tid < D) {
    double2 t = make_double2(0.0, 0.0);
    for (int h = 0; h < G; h++) {
      t.x += shares[tid * G + h].x;
      t.y += shares[tid * G + h].y;
    }
    partials[(size_t)blockIdx.x * 64 + tid] = t;
  }
}

// Reverse step of a register that is one tile (p.pos: physical bits), in one CTA.  gdst: 2 * 2^nk doubles or nullptr.
__global__ void __launch_bounds__(QDC_DIAGK_NT)
    k_diag_k_rev_whole(cplx_t* __restrict__ fwd, cplx_t* __restrict__ bwd, const cplx_t* __restrict__ A,
                       const cplx_t* __restrict__ B, const DiagKPos p, int n_loc, double* __restrict__ gdst) {
  constexpr int NT = QDC_DIAGK_NT;
  __shared__ cplx_t As[64], Bs[64];
  __shared__ double2 shares[NT];
  const int tid = threadIdx.x, N = 1 << n_loc;
  for (int i = tid; i < (1 << p.nk); i += NT) {
    As[i] = A[i];
    Bs[i] = B[i];
  }
  __syncthreads();
  for (int e = tid; e < N; e += NT) diag_k_mul(As[diag_k_index((uint64_t)e, p)], fwd[e].x, fwd[e].y);
  __syncthreads();
  if (gdst) {
    const int D = 1 << p.nk, G = NT / D, bin = tid / G, g = tid % G, nrest = N >> p.nk;
    double2 sum = make_double2(0.0, 0.0);
    for (int r = g; r < nrest; r += G) {
      const int e = diag_k_deposit(bin, r, p, n_loc);
      const cplx_t f = fwd[e], b = bwd[e];
      sum.x += (double)(b.x * f.x - b.y * f.y);
      sum.y += (double)(b.x * f.y + b.y * f.x);
    }
    shares[tid] = sum;
    __syncthreads();
    if (tid < D) {
      double2 t = make_double2(0.0, 0.0);
      for (int h = 0; h < G; h++) {
        t.x += shares[tid * G + h].x;
        t.y += shares[tid * G + h].y;
      }
      gdst[2 * tid] = t.x;
      gdst[2 * tid + 1] = t.y;
    }
    __syncthreads();
  }
  for (int e = tid; e < N; e += NT) diag_k_mul(Bs[diag_k_index((uint64_t)e, p)], bwd[e].x, bwd[e].y);
}

// ------------------------------------------------------------ host side
// Appends the device forms of the diagonal d of instruction `in` (2^k entries), folded over this rank's bits at the
// physical positions pk of its plan step, to `h`:  forward: d;  reverse: the un-compute form (conj d, or 1 / d in
// double precision for NonU gates), then d.  A zero entry of a NonU gate fails with the text of the inverse.
inline const char* Circuit::diag_k_forms(const cplx_t* d, const Inst& in, const int* pk, bool reverse,
                                         std::vector<cplx_t>* h) {
  const int D = 1 << in.nk;
  const qdc::DiagFold f = qdc::diag_fold_split(pk, in.nk, n_loc_, rank_);
  std::vector<cplx_t> loc;
  if (reverse) {
    std::vector<cplx_t> inv(D);
    for (int j = 0; j < D; j++) {
      if (kind_is_nonu(in.kind)) {
        const zc v(d[j].x, d[j].y);
        if (v == zc(0, 0)) return qdc_errf("U(%d, %d) is zero.", j + 1, j + 1);
        const zc w = zc(1, 0) / v;
        inv[j].x = (real_t)w.real();
        inv[j].y = (real_t)w.imag();
      } else {
        inv[j].x = d[j].x;
        inv[j].y = -d[j].y;
      }
    }
    qdc::diag_fold(f, in.nk, inv.data(), &loc);
    h->insert(h->end(), loc.begin(), loc.end());
  }
  qdc::diag_fold(f, in.nk, d, &loc);
  h->insert(h->end(), loc.begin(), loc.end());
  return nullptr;
}

inline const char* Circuit::launch_diag_k(cplx_t* buf, const cplx_t* form, const DiagKPos& p) {
  static thread_local int bps = 0;
  DeviceInfo di;
  QDC_TRY(qdc_device_info(&di));
  if (bps == 0) QDC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, k_diag_k, QDC_BLOCK, 0));
  const uint64_t nvec = 1ull << (n_loc_ - QDC_LV);
  const int grid = pick_grid(nvec, QDC_DIAGK_UNROLL, bps, di.sm_count);
  k_diag_k<<<grid, QDC_BLOCK, 0, stream_>>>((vec_t*)buf, form, p, nvec);
  QDC_CUDA(cudaGetLastError());
  return nullptr;
}

// the k_loc local positions of a diagonal k-qubit step on this rank (physical bits)
static inline DiagKPos diag_k_local(const qdc::DiagFold& f) {
  DiagKPos p;
  p.nk = f.k_loc;
  for (int q = 0; q < 6; q++) p.pos[q] = f.loc[q];
  return p;
}

// buf <- (form on the step's positions) buf: the forward pass, and the un-compute while no adjoint exists
inline const char* Circuit::diag_k_apply(const qdc::Step& st, cplx_t* buf, const cplx_t* form, int cat) {
  const DiagKPos p = diag_k_local(qdc::diag_fold_split(st.pk, st.nk, n_loc_, rank_));
  PROF(cat, 2, launch_diag_k(buf, form, p));
  account(1, 1, 2);
  return nullptr;
}

inline const char* Circuit::launch_diag_k_rev_whole(const DiagKPos& p, const cplx_t* A, const cplx_t* B,
                                                    double* gdst) {
  k_diag_k_rev_whole<<<1, QDC_DIAGK_NT, 0, stream_>>>(state_, bwd_, A, B, p, n_loc_, gdst);
  QDC_CUDA(cudaGetLastError());
  return nullptr;
}

template <int NI>
inline const char* Circuit::launch_diag_k_rev(const DensKParams& dp, const DiagKPos& p, const cplx_t* A,
                                              const cplx_t* B, double* gdst) {
  const size_t smem = gdst ? sizeof(double2) * NI * QDC_VA * QDC_DIAGK_NT : 0;
  int grid = 0;
  QDC_TRY(tile_grid((const void*)k_diag_k_rev<NI>, QDC_DIAGK_NT, smem, dp.geo.ntiles, &grid));
  const size_t need = (size_t)grid * 64 * 2;
  if (gdst && need > tile_partials_cap_) {
    if (tile_partials_) QDC_CUDA(cudaFree(tile_partials_));
    QDC_CUDA(cudaMalloc((void**)&tile_partials_, need * sizeof(double)));
    tile_partials_cap_ = need;
  }
  k_diag_k_rev<NI><<<grid, QDC_DIAGK_NT, smem, stream_>>>((vec_t*)state_, (vec_t*)bwd_, A, B, dp.geo, p,
                                                           gdst ? (double2*)tile_partials_ : nullptr);
  QDC_CUDA(cudaGetLastError());
  if (gdst) {
    k_diag_k_final<<<1 << p.nk, 256, 0, stream_>>>((const double2*)tile_partials_, grid, gdst);
    QDC_CUDA(cudaGetLastError());
  }
  return nullptr;
}

// reverse step with an adjoint; gdst: the 2^k_loc gradient entries (2 doubles each) of a variable gate, nullptr for
// a constant one (scattered to the gate's 2^k entries by the caller)
inline const char* Circuit::diag_k_reverse(const qdc::Step& st, const cplx_t* A, const cplx_t* B, double* gdst) {
  const qdc::DiagFold f = qdc::diag_fold_split(st.pk, st.nk, n_loc_, rank_);
  DiagKPos p = diag_k_local(f);
  const int cat = CAT_DIAG_K_REV;
  if (n_loc_ <= QDC_LV + 11) {   // the register fits one tile
    PROF(cat, 4, launch_diag_k_rev_whole(p, A, B, gdst));
  } else {
    static thread_local DensKParams dp;
    qdc::Step ls = st;
    ls.nk = f.k_loc;
    for (int q = 0; q < 6; q++) ls.pk[q] = f.loc[q];
    QDC_TRY(fill_dens_k_params(ls, &dp));
    for (int q = 0; q < p.nk; q++) p.pos[q] = dp.a[q];   // tile-local bits
    const int ni = 1 << (dp.geo.T - QDC_LV - 8);
    switch (ni) {
      case 4: PROF(cat, 4, launch_diag_k_rev<4>(dp, p, A, B, gdst)); break;
      case 8: PROF(cat, 4, launch_diag_k_rev<8>(dp, p, A, B, gdst)); break;
      default: return qdc_errf("internal: diagonal k-qubit gate on a %d-bit tile.", dp.geo.T);
    }
  }
  account(gdst && n_loc_ > QDC_LV + 11 ? 2 : 1, 2, 4);
  return nullptr;
}
