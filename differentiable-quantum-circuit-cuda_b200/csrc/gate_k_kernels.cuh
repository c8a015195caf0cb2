// k-qubit gates (3 <= k <= 6) and their reverse steps (kinds CONST_GATE_K / VAR_GATE_K / *_NONU).
//
//   k_gate_k     : psi[r, rest] = sum_c A[r, c] psi[c, rest]                        (2*S, in place)
//   k_gate_k_rev : fwd <- A fwd;  G[r, c] (=)= sum_rest bwd[r, rest] fwd[c, rest];  bwd <- B bwd   (4*S)
// with r, c the k-bit index over `positions` (positions[0] is the most significant bit).  k_gate_k applies U in the
// forward pass and the un-compute form (U^dagger, or U^-1 for NonU gates) in the reverse pass while no adjoint exists;
// k_gate_k_rev is the reverse step of the reference at width k: A = the un-compute form, the gradient of q2grad
// (no conjugation) from the un-computed state and the adjoint before the pull-back, B = U^T.
//
// Both kernels walk the tiles of k_dens_k / k_seed_k (fill_dens_k_params, dens_k_kernels.cuh) and re-stage a tile
// as a D x (rest + 1) matrix.  The matrices come from device memory (every k-gate matrix of a call is uploaded in
// one copy) and are staged in shared memory once per CTA, transposed: As[c D + r] = A[r, c], so the reads of a warp
// (consecutive rest columns, one row block) are broadcasts.  Every tile element is written once per sweep.
// The reverse step keeps ONE raw tile buffer: the state tile is loaded, staged, un-computed into the raw buffer,
// stored and re-staged before the adjoint tile is loaded into the same buffer.  Its shared memory is one raw tile,
// two staged tiles and two D x D matrices: 231,808 bytes for k = 6 in f64 (227 KiB allow 232,448), 165,376 in f32.
// The gradient is summed like a density: real_t per tile, double across the CTA's tiles, then a fixed-order sum over
// (CTA, share) in k_dens_k_final -- no floating-point atomics, the same result run to run.
#pragma once
#include <complex>
#include <vector>

#include "dens_k_kernels.cuh"

// X[roff[r] | resto[j]] = sum_c As[c D + r] Y[c ld + j]: the item loop of k_seed_k without the seed's accumulation
template <int KQ>
__device__ __forceinline__ void gate_k_matvec(const cplx_t* As, const cplx_t* Y, int ld, int nrest, cplx_t* X,
                                              const int* roff, const int* resto) {
  constexpr int D = 1 << KQ, Q = D / 4;
  // items: (row block rb, rest columns jb + js l), consecutive threads on consecutive jb (As reads broadcast)
  const int nj = nrest >= 4 ? nrest / 4 : 1, js = nj, nitems = Q * nj;
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
      for (int i = 0; i < 4; i++) g[i] = As[c * D + rb + Q * i];
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
        if (j < nrest) X[roff[rb + Q * i] | resto[j]] = acc[i][l];   // written by this thread only
      }
  }
}

// acc[2 (4 i + l) + re/im] += sum over this share's rest columns of Yb[rb + Q i, j] Yf[cb + Q l, j]
template <int KQ>
__device__ __forceinline__ void gate_k_grad_items(const cplx_t* Yb, const cplx_t* Yf, int ld, int nrest, int s, int rb,
                                                  int cb, real_t (&acc)[32]) {
  constexpr int Q = (1 << KQ) / 4, S = QDC_DENSK_NT / (Q * Q);
  for (int j = s; j < nrest; j += S) {
    cplx_t a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {
      a[i] = Yb[(rb + Q * i) * ld + j];
      b[i] = Yf[(cb + Q * i) * ld + j];
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
#pragma unroll
      for (int l = 0; l < 4; l++) {  // a b, no conjugation
        acc[2 * (4 * i + l)] += a[i].x * b[l].x - a[i].y * b[l].y;
        acc[2 * (4 * i + l) + 1] += a[i].x * b[l].y + a[i].y * b[l].x;
      }
    }
  }
}

__device__ __forceinline__ void gate_k_store(const DensKParams& p, const TileAddr<QDC_DENSK_NT>& ta, cplx_t* gmem,
                                             cplx_t* sm, uint64_t tile) {
  if (p.whole) {
    for (int i = threadIdx.x; i < (1 << p.geo.T); i += QDC_DENSK_NT) gmem[i] = sm[i];
  } else {
    tile_io<QDC_DENSK_NT, false>((vec_t*)gmem, (vec_t*)sm, ta, p.geo.tile(tile) >> QDC_LV);
  }
}

// buf <- (A on the positions) buf;  At: A transposed (At[c D + r] = A[r, c]), in global memory
template <int KQ>
__global__ void __launch_bounds__(QDC_DENSK_NT, 1)
    k_gate_k(cplx_t* __restrict__ buf, const cplx_t* __restrict__ At, const __grid_constant__ DensKParams p) {
  constexpr int D = 1 << KQ;
  extern __shared__ __align__(16) unsigned char gatek_smem[];
  const int T = p.geo.T, nrest = 1 << (T - KQ), ld = nrest + 1;
  cplx_t* X = (cplx_t*)gatek_smem;
  cplx_t* Y = X + (1 << T);
  cplx_t* As = Y + D * ld;
  int* roff = (int*)(As + D * D);
  int* resto = roff + D;
  dens_k_tables<KQ>(p, roff, resto);
  for (int i = threadIdx.x; i < D * D; i += QDC_DENSK_NT) As[i] = At[i];
  TileAddr<QDC_DENSK_NT> ta;
  if (!p.whole) ta.init(p.geo);
  const uint64_t ntiles = p.whole ? 1 : p.geo.ntiles;
  for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    dens_k_load(p, ta, buf, X, tile);
    __syncthreads();
    dens_k_stage<KQ, false>(X, Y, roff, resto, T, ld);
    __syncthreads();
    gate_k_matvec<KQ>(As, Y, ld, nrest, X, roff, resto);
    __syncthreads();
    gate_k_store(p, ta, buf, X, tile);
    __syncthreads();
  }
}

// Reverse step: fwd <- A fwd, then (partials != nullptr) the gradient partials of bwd (x) fwd, then bwd <- B bwd.
// At / Bt transposed like k_gate_k's.  partials: [gridDim.x][QDC_DENSK_NT][32] doubles, summed by k_dens_k_final.
template <int KQ>
__global__ void __launch_bounds__(QDC_DENSK_NT, 1)
    k_gate_k_rev(cplx_t* __restrict__ fwd, cplx_t* __restrict__ bwd, const cplx_t* __restrict__ At,
                 const cplx_t* __restrict__ Bt, const __grid_constant__ DensKParams p, double* __restrict__ partials) {
  constexpr int D = 1 << KQ, Q = D / 4, OWN = Q * Q;
  extern __shared__ __align__(16) unsigned char gatek_smem[];
  const int T = p.geo.T, nrest = 1 << (T - KQ), ld = nrest + 1;
  cplx_t* X = (cplx_t*)gatek_smem;
  cplx_t* Yf = X + (1 << T);
  cplx_t* Yb = Yf + D * ld;
  cplx_t* As = Yb + D * ld;
  cplx_t* Bs = As + D * D;
  int* roff = (int*)(Bs + D * D);
  int* resto = roff + D;
  dens_k_tables<KQ>(p, roff, resto);
  for (int i = threadIdx.x; i < D * D; i += QDC_DENSK_NT) {
    As[i] = At[i];
    Bs[i] = Bt[i];
  }
  TileAddr<QDC_DENSK_NT> ta;
  if (!p.whole) ta.init(p.geo);
  const int o = threadIdx.x % OWN, s = threadIdx.x / OWN, rb = o / Q, cb = o % Q;
  double dacc[32];
#pragma unroll
  for (int q = 0; q < 32; q++) dacc[q] = 0.0;
  const uint64_t ntiles = p.whole ? 1 : p.geo.ntiles;
  for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    // un-compute the state tile and keep it staged (Yf) for the gradient
    dens_k_load(p, ta, fwd, X, tile);
    __syncthreads();
    dens_k_stage<KQ, false>(X, Yf, roff, resto, T, ld);
    __syncthreads();
    gate_k_matvec<KQ>(As, Yf, ld, nrest, X, roff, resto);
    __syncthreads();
    gate_k_store(p, ta, fwd, X, tile);
    dens_k_stage<KQ, false>(X, Yf, roff, resto, T, ld);
    __syncthreads();
    // the adjoint tile: gradient, then the pull-back
    dens_k_load(p, ta, bwd, X, tile);
    __syncthreads();
    dens_k_stage<KQ, false>(X, Yb, roff, resto, T, ld);
    __syncthreads();
    if (partials) {
#ifdef QDC_F64
      gate_k_grad_items<KQ>(Yb, Yf, ld, nrest, s, rb, cb, dacc);
#else
      real_t acc[32];
#pragma unroll
      for (int q = 0; q < 32; q++) acc[q] = 0;
      gate_k_grad_items<KQ>(Yb, Yf, ld, nrest, s, rb, cb, acc);
#pragma unroll
      for (int q = 0; q < 32; q++) dacc[q] += (double)acc[q];
#endif
    }
    gate_k_matvec<KQ>(Bs, Yb, ld, nrest, X, roff, resto);
    __syncthreads();
    gate_k_store(p, ta, bwd, X, tile);
    __syncthreads();
  }
  if (partials) {
    double* dst = partials + ((size_t)blockIdx.x * QDC_DENSK_NT + threadIdx.x) * 32;
#pragma unroll
    for (int q = 0; q < 32; q++) dst[q] = dacc[q];
  }
}

// ------------------------------------------------------------ host side
// Gauss-Jordan inverse with partial pivoting in double precision, on the heap (a 64 x 128 complex work matrix is
// 128 KiB): engine.cuh's `invert` at run-time size, with the same error text for a singular pivot.
static inline const char* invert_k(std::vector<zc>& m, int K) {
  const int W = 2 * K;
  std::vector<zc> a((size_t)K * W);
  for (int r = 0; r < K; r++)
    for (int c = 0; c < K; c++) {
      a[(size_t)r * W + c] = m[(size_t)r * K + c];
      a[(size_t)r * W + K + c] = (r == c) ? zc(1, 0) : zc(0, 0);
    }
  for (int col = 0; col < K; col++) {
    int piv = col;
    double best = std::abs(a[(size_t)col * W + col]);
    for (int r = col + 1; r < K; r++)
      if (std::abs(a[(size_t)r * W + col]) > best) {
        best = std::abs(a[(size_t)r * W + col]);
        piv = r;
      }
    if (best == 0.0) return qdc_errf("U(%d, %d) is zero.", col + 1, col + 1);
    if (piv != col)
      for (int c = 0; c < W; c++) std::swap(a[(size_t)piv * W + c], a[(size_t)col * W + c]);
    const zc inv = zc(1, 0) / a[(size_t)col * W + col];
    for (int c = 0; c < W; c++) a[(size_t)col * W + c] *= inv;
    for (int r = 0; r < K; r++) {
      if (r == col) continue;
      const zc f = a[(size_t)r * W + col];
      if (f == zc(0, 0)) continue;
      for (int c = 0; c < W; c++) a[(size_t)r * W + c] -= f * a[(size_t)col * W + c];
    }
  }
  for (int r = 0; r < K; r++)
    for (int c = 0; c < K; c++) m[(size_t)r * K + c] = a[(size_t)r * W + K + c];
  return nullptr;
}

// Appends the device forms of k-gate matrix U (D x D, row-major) to `h`, each transposed for the kernels:
// forward: U;  reverse: the un-compute form (U^dagger, or U^-1 for NonU gates), then U^T.
inline const char* Circuit::gate_k_forms(const cplx_t* U, int nk, bool nonu, bool reverse, std::vector<cplx_t>* h) {
  const int D = 1 << nk;
  const size_t base = h->size();
  h->resize(base + (reverse ? 2 : 1) * (size_t)D * D);
  cplx_t* out = h->data() + base;
  if (!reverse) {
    for (int r = 0; r < D; r++)
      for (int c = 0; c < D; c++) out[c * D + r] = U[r * D + c];
    return nullptr;
  }
  if (nonu) {
    std::vector<zc> m((size_t)D * D);
    for (int i = 0; i < D * D; i++) m[i] = zc(U[i].x, U[i].y);
    QDC_TRY(invert_k(m, D));
    for (int r = 0; r < D; r++)
      for (int c = 0; c < D; c++) {
        const zc v = m[(size_t)r * D + c];
        out[c * D + r].x = (real_t)v.real();
        out[c * D + r].y = (real_t)v.imag();
      }
  } else {
    for (int i = 0; i < D * D; i++) {   // (U^dagger)^T = conj U
      out[i].x = U[i].x;
      out[i].y = -U[i].y;
    }
  }
  for (int i = 0; i < D * D; i++) out[D * D + i] = U[i];   // (U^T)^T = U
  return nullptr;
}

template <int KQ>
static inline size_t gate_k_rev_smem(int T) {
  constexpr int D = 1 << KQ;
  const int nrest = 1 << (T - KQ);
  return (sizeof(cplx_t) << T) + 2 * sizeof(cplx_t) * D * (nrest + 1) + 2 * sizeof(cplx_t) * D * D +
         sizeof(int) * (D + nrest);
}

template <int KQ>
inline const char* Circuit::launch_gate_k(const DensKParams& p, cplx_t* buf, const cplx_t* At) {
  const size_t smem = dens_k_smem<KQ>(p.geo.T, true);   // the seed's layout: raw tile, staged tile, one matrix
  int grid = 0;
  QDC_TRY(tile_grid((const void*)k_gate_k<KQ>, QDC_DENSK_NT, smem, p.whole ? 1 : p.geo.ntiles, &grid));
  k_gate_k<KQ><<<grid, QDC_DENSK_NT, smem, stream_>>>(buf, At, p);
  QDC_CUDA(cudaGetLastError());
  return nullptr;
}

template <int KQ>
inline const char* Circuit::launch_gate_k_rev(const DensKParams& p, const cplx_t* At, const cplx_t* Bt,
                                              double* gdst) {
  constexpr int OWN = (1 << KQ) / 4 * ((1 << KQ) / 4), S = QDC_DENSK_NT / OWN;
  const size_t smem = gate_k_rev_smem<KQ>(p.geo.T);
  int grid = 0;
  QDC_TRY(tile_grid((const void*)k_gate_k_rev<KQ>, QDC_DENSK_NT, smem, p.whole ? 1 : p.geo.ntiles, &grid));
  const size_t need = (size_t)grid * QDC_DENSK_NT * 32;
  if (gdst && need > tile_partials_cap_) {
    if (tile_partials_) QDC_CUDA(cudaFree(tile_partials_));
    QDC_CUDA(cudaMalloc((void**)&tile_partials_, need * sizeof(double)));
    tile_partials_cap_ = need;
  }
  k_gate_k_rev<KQ><<<grid, QDC_DENSK_NT, smem, stream_>>>(state_, bwd_, At, Bt, p, gdst ? tile_partials_ : nullptr);
  QDC_CUDA(cudaGetLastError());
  if (gdst) {
    k_dens_k_final<KQ><<<OWN, 256, 0, stream_>>>(tile_partials_, grid * S, gdst);
    QDC_CUDA(cudaGetLastError());
  }
  return nullptr;
}

// buf <- (At^T on the step's positions) buf: the forward pass, and the un-compute while no adjoint exists
inline const char* Circuit::gate_k_apply(const qdc::Step& st, cplx_t* buf, const cplx_t* At, int cat) {
  static thread_local DensKParams p;
  QDC_TRY(fill_dens_k_params(st, &p));
  switch (st.nk) {
    case 3: PROF(cat, 2, launch_gate_k<3>(p, buf, At)); break;
    case 4: PROF(cat, 2, launch_gate_k<4>(p, buf, At)); break;
    case 5: PROF(cat, 2, launch_gate_k<5>(p, buf, At)); break;
    case 6: PROF(cat, 2, launch_gate_k<6>(p, buf, At)); break;
    default: return qdc_errf("internal: %d-qubit gate step.", st.nk);
  }
  account(1, 1, 2);
  return nullptr;
}

// reverse step with an adjoint; gdst: the gradient (2 * 4^k doubles) of a variable gate, nullptr for a constant one
inline const char* Circuit::gate_k_reverse(const qdc::Step& st, const cplx_t* At, const cplx_t* Bt, double* gdst) {
  static thread_local DensKParams p;
  QDC_TRY(fill_dens_k_params(st, &p));
  switch (st.nk) {
    case 3: PROF(CAT_GATE_K_REV, 4, launch_gate_k_rev<3>(p, At, Bt, gdst)); break;
    case 4: PROF(CAT_GATE_K_REV, 4, launch_gate_k_rev<4>(p, At, Bt, gdst)); break;
    case 5: PROF(CAT_GATE_K_REV, 4, launch_gate_k_rev<5>(p, At, Bt, gdst)); break;
    case 6: PROF(CAT_GATE_K_REV, 4, launch_gate_k_rev<6>(p, At, Bt, gdst)); break;
    default: return qdc_errf("internal: %d-qubit gate step.", st.nk);
  }
  account(gdst ? 2 : 1, 2, 4);
  return nullptr;
}
