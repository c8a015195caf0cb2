// Circuit executor: the B200 counterpart of the reference's Rust `Circuit`
// (/root/reference/src/circuit.rs:86-430) and `QuantizedTensor`
// (src/quantized_tensor.rs:54-238), behind the C ABI of include/qdc_circuit.h.
//
// Differences that matter on B200 (design, not semantics):
//  * two resident 2^n buffers (state + adjoint) instead of four
//    (src/circuit.rs:96-102, 276, 396-398): |0..0> is generated, not stored,
//    and the density seed is fused so no transient `bwd_addition` exists;
//  * every density / gradient lands in one device-resident double buffer that
//    is copied back ONCE per call (the reference does cudaMalloc + blocking
//    D2H + cudaFree per gradient, src/primitives.cu:264-291);
//  * the backward step of a gate is one 4*S kernel (engine.cuh) instead of
//    three 2*S kernels (src/circuit.rs:320-333).
#pragma once
#include <algorithm>
#include <string>
#include <vector>

#include "diag_k_host.hpp"
#include "engine.cuh"
#include "nccl_dyn.hpp"
#include "scheduler.hpp"
#ifndef QDC_F64
#include "tc_block.cuh"
#endif

enum Kind {
  K_CONST_Q2 = 0, K_VAR_Q2, K_CONST_Q2_NONU, K_VAR_Q2_NONU, K_CONST_Q2_DIAG, K_VAR_Q2_DIAG,
  K_CONST_Q1, K_CONST_Q1_NONU, K_VAR_Q1, K_VAR_Q1_NONU,
  K_Q2_DENS, K_Q1_DENS, K_DIFF_Q2_DENS, K_DIFF_Q1_DENS,
  K_DENS_K, K_DIFF_DENS_K,  // densities on 3..6 qubits (add_dens; dens_k_kernels.cuh)
  K_CONST_GATE_K, K_VAR_GATE_K, K_CONST_GATE_K_NONU, K_VAR_GATE_K_NONU,  // gates on 3..6 qubits (add_gate; gate_k_kernels.cuh)
  K_CONST_DIAG_K, K_VAR_DIAG_K, K_CONST_DIAG_K_NONU, K_VAR_DIAG_K_NONU   // diagonal gates on 1..6 qubits (add_gate_diag;
                                                                         // diag_k_kernels.cuh)
};

// one- and two-qubit gates (the k-qubit gates are kind_is_k_gate)
static inline bool kind_is_gate(int k) { return k <= K_VAR_Q1_NONU; }
static inline bool kind_is_var(int k) {
  return k == K_VAR_Q2 || k == K_VAR_Q2_NONU || k == K_VAR_Q2_DIAG || k == K_VAR_Q1 || k == K_VAR_Q1_NONU ||
         k == K_VAR_GATE_K || k == K_VAR_GATE_K_NONU || k == K_VAR_DIAG_K || k == K_VAR_DIAG_K_NONU;
}
static inline bool kind_is_nonu(int k) {
  return k == K_CONST_Q2_NONU || k == K_VAR_Q2_NONU || k == K_CONST_Q1_NONU || k == K_VAR_Q1_NONU ||
         k == K_CONST_GATE_K_NONU || k == K_VAR_GATE_K_NONU || k == K_CONST_DIAG_K_NONU || k == K_VAR_DIAG_K_NONU;
}
static inline bool kind_is_diag(int k) { return k == K_CONST_Q2_DIAG || k == K_VAR_Q2_DIAG; }
static inline bool kind_is_q1(int k) { return k >= K_CONST_Q1 && k <= K_VAR_Q1_NONU; }
static inline bool kind_is_q2dense(int k) { return k <= K_VAR_Q2_NONU; }
static inline bool kind_is_dens(int k) { return k >= K_Q2_DENS && k <= K_DIFF_DENS_K; }
static inline bool kind_is_k_gate(int k) { return k >= K_CONST_GATE_K && k <= K_VAR_GATE_K_NONU; }
static inline bool kind_is_diag_k(int k) { return k >= K_CONST_DIAG_K && k <= K_VAR_DIAG_K_NONU; }
static inline bool kind_is_diff_dens(int k) { return k == K_DIFF_Q2_DENS || k == K_DIFF_Q1_DENS || k == K_DIFF_DENS_K; }
static inline bool kind_is_k_dens(int k) { return k == K_DENS_K || k == K_DIFF_DENS_K; }
static inline bool kind_is_q1_dens(int k) { return k == K_Q1_DENS || k == K_DIFF_Q1_DENS; }
static inline int kind_gate_len(int k) { return kind_is_q2dense(k) ? 16 : 4; }
static inline int kind_dens_len(int k) { return kind_is_q1_dens(k) ? 4 : 16; }

struct Inst {
  int kind;
  int pos2, pos1;  // q1 kinds use pos2 only
  int nk = 0;      // k-qubit densities and gates (dense, diagonal): the qubits kpos[0..nk-1], most significant first (pos2 = pos1 = -1)
  int kpos[6] = {-1, -1, -1, -1, -1, -1};
};

// complex entries of a density's output / cotangent
static inline size_t dens_len(const Inst& in) {
  return kind_is_k_dens(in.kind) ? (size_t)1 << (2 * in.nk) : (size_t)kind_dens_len(in.kind);
}

// complex entries of a gate's matrix / gradient
static inline size_t gate_len(const Inst& in) {
  if (kind_is_diag_k(in.kind)) return (size_t)1 << in.nk;
  return kind_is_k_gate(in.kind) ? (size_t)1 << (2 * in.nk) : (size_t)kind_gate_len(in.kind);
}

struct Stats {
  uint64_t kernel_launches = 0, hbm_passes = 0, algorithmic_bytes = 0;
};

struct DensGroup;
struct TileDensParams;
struct DensKParams;
struct DiagKPos;
struct TcState;
struct TcPass;

struct GateList {
  const cplx_t* flat;
  const uint32_t* lens;
  size_t count;
};

// Per-category device timing with CUDA events on the executing stream
// (enabled by option "profile"); feeds bench.py's roofline block.
enum ProfCat {
  CAT_FWD_Q1 = 0, CAT_FWD_Q2, CAT_FWD_DIAG, CAT_DENSITY, CAT_SEED, CAT_UNCOMPUTE, CAT_REV_Q1, CAT_REV_Q2,
  CAT_REV_DIAG, CAT_REV_CONST, CAT_TILE_FWD, CAT_TILE_BWD, CAT_EXCHANGE, CAT_TC_FWD, CAT_TC_BWD, CAT_GATE_K_FWD,
  CAT_GATE_K_REV, CAT_DIAG_K_FWD, CAT_DIAG_K_REV, CAT_COUNT
};
static const char* const kProfCatNames[CAT_COUNT] = {
    "fwd_q1", "fwd_q2", "fwd_diag", "density", "seed", "uncompute", "rev_q1", "rev_q2",
    "rev_diag", "rev_const", "tile_fwd", "tile_bwd", "exchange", "tc_fwd", "tc_bwd", "gate_k_fwd", "gate_k_rev",
    "diag_k_fwd", "diag_k_rev"};

struct ProfEntry {
  uint64_t launches = 0;
  double ms = 0;
  uint64_t alg_bytes = 0;
};

struct Profiler {
  bool on = false;
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  struct Rec { int cat; cudaEvent_t a, b; uint64_t bytes; };
  std::vector<Rec> recs;
  ProfEntry cats[CAT_COUNT];
  cudaEvent_t get() {
    if (used == pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    return pool[used++];
  }
  void reset() {
    used = 0;
    recs.clear();
    for (auto& c : cats) c = ProfEntry();
  }
  cudaEvent_t begin(cudaStream_t st) {
    cudaEvent_t a = get();
    cudaEventRecord(a, st);
    return a;
  }
  void end(cudaStream_t st, int cat, cudaEvent_t a, uint64_t bytes) {
    cudaEvent_t b = get();
    cudaEventRecord(b, st);
    recs.push_back(Rec{cat, a, b, bytes});
  }
  void collect() {  // after the stream has been synchronised
    for (const Rec& r : recs) {
      float ms = 0;
      cudaEventElapsedTime(&ms, r.a, r.b);
      cats[r.cat].launches++;
      cats[r.cat].ms += ms;
      cats[r.cat].alg_bytes += r.bytes;
    }
    recs.clear();
    used = 0;
  }
  ~Profiler() {
    for (cudaEvent_t e : pool) cudaEventDestroy(e);
  }
};

// PROF(cat, algorithmic passes, launch expression)
#define PROF(cat, alg_passes, expr)                                           \
  do {                                                                        \
    cudaEvent_t pa_ = nullptr;                                                \
    if (prof_.on) pa_ = prof_.begin(stream_);                                 \
    QDC_TRY(expr);                                                            \
    if (prof_.on) prof_.end(stream_, cat, pa_, (uint64_t)(alg_passes) * bytes()); \
  } while (0)

// ---- half-shard pack / unpack for qubit-remap exchanges ------------------
// dst[i] = src[i with bit `pos` forced to `val`]  (gather), or the inverse.
template <typename V, bool GATHER>
__global__ void __launch_bounds__(QDC_BLOCK)
    k_half_copy(V* __restrict__ full, V* __restrict__ half, int pos, int val, uint64_t nhalf) {
  const uint64_t stride = (uint64_t)gridDim.x * QDC_BLOCK;
  for (uint64_t i = (uint64_t)blockIdx.x * QDC_BLOCK + threadIdx.x; i < nhalf; i += stride) {
    const uint64_t j = ins0(i, pos) | ((uint64_t)val << pos);
    if (GATHER) half[i] = full[j]; else full[j] = half[i];
  }
}

// ---- qubit-remap swap fused with the exchange, over NVLink peer memory -----
// new[lpos = b, rank bit = c] = old[lpos = c, rank bit = b]: the element
// (lpos = 1-c, x) of this rank trades places with the element (lpos = c, x) of
// the partner.  Every such PAIR is owned by exactly one of the two GPUs (the
// x range is split in halves by rank bit), which loads both elements -- the
// partner's through its peer mapping -- and stores them swapped.  No staging
// buffer, no pack / unpack passes, in place on both GPUs, and no thread ever
// waits on the other GPU (ordering is by stream-ordered token exchanges
// before and after the kernel).
template <typename V>
__global__ void __launch_bounds__(QDC_BLOCK)
    k_peer_swap(V* __restrict__ mine, V* __restrict__ peer, int pos, int c, uint64_t x_begin, uint64_t x_end) {
  const uint64_t stride = (uint64_t)gridDim.x * QDC_BLOCK;
  constexpr int U = 4;
  for (uint64_t x0 = x_begin + (uint64_t)blockIdx.x * QDC_BLOCK + threadIdx.x; x0 < x_end; x0 += stride * U) {
    V a[U], b[U];
    uint64_t mi[U], pi[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t x = x0 + (uint64_t)u * stride;
      const uint64_t base = ins0(x, pos);
      mi[u] = base | ((uint64_t)(1 - c) << pos);
      pi[u] = base | ((uint64_t)c << pos);
      if (x < x_end) {
        a[u] = mine[mi[u]];
        b[u] = peer[pi[u]];
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t x = x0 + (uint64_t)u * stride;
      if (x < x_end) {
        mine[mi[u]] = b[u];
        peer[pi[u]] = a[u];
      }
    }
  }
}

// ---- several (global qubit <-> local position) swaps in ONE exchange --------
// The scheduler's remaps come in runs (35 q on 8 ranks: g0 <-> l4, g1 <-> l5, g2 <-> l6 back to back).  k swaps carried
// out one after the other move k halves of the shard; done at once,
//   new[local bits = b, rank bits = c] = old[local bits = c, rank bits = b]       (b, c: k-bit values),
// this rank keeps the 2^-k of its shard with b == c and trades one 2^-k with each of the 2^k - 1 ranks of its group:
// (1 - 2^-k) of a shard instead of k / 2 (7/8 instead of 3/2 for k = 3), all partners at once through the NVSwitch.
// Element (local bits = b, x) of this rank trades places with element (local bits = c, x) of the rank whose selected
// bits are b; of the two owners of such a pair the one with the smaller selected value handles the lower half of the
// x range, the other one the upper half.
struct MultiSwapArgs {
  int k;                  // swapped pairs (2 or 3)
  int pos_sorted[3];      // vector-index bit positions of the local qubits, ascending (zero insertion)
  int pos_pair[3];        // ... in pair order: bit i of a selected value <-> pos_pair[i]
  int c;                  // selected value of this rank
  int half_log2;          // log2 of the x range each side owns per partner
  void* peer[8];          // [b]: the same buffer on the rank whose selected bits are b
};

template <typename V>
__global__ void __launch_bounds__(QDC_BLOCK) k_peer_multiswap(V* __restrict__ mine, const MultiSwapArgs a) {
  const uint64_t stride = (uint64_t)gridDim.x * QDC_BLOCK;
  const uint64_t per = 1ull << a.half_log2, total = per * (uint64_t)((1 << a.k) - 1);
  constexpr int U = 4;
  int dep_c = 0;
  for (int i = 0; i < a.k; i++) dep_c |= ((a.c >> i) & 1) << a.pos_pair[i];
  for (uint64_t w0 = (uint64_t)blockIdx.x * QDC_BLOCK + threadIdx.x; w0 < total; w0 += stride * U) {
    V va[U], vb[U];
    uint64_t mi[U], pi[U];
    V* pp[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t w = w0 + (uint64_t)u * stride;
      if (w < total) {
        // partner of phase j: c XOR (j + 1) -- a perfect matching of the group in every phase, so each rank trades with
        // exactly one partner at a time, both ways.  (Enumerating "every value but c" in ascending order sent two ranks
        // to the same partner at once: 371 instead of 695 GB/s per direction, profiles/r2_bench_8gpu_35q_multiswap_v1.json.)
        const int j = (int)(w >> a.half_log2);
        const int b = a.c ^ (j + 1);
        uint64_t x = (w & (per - 1ull)) + (a.c < b ? 0ull : per);
        for (int i = 0; i < a.k; i++) x = ins0(x, a.pos_sorted[i]);
        uint64_t dep_b = 0;
        for (int i = 0; i < a.k; i++) dep_b |= (uint64_t)((b >> i) & 1) << a.pos_pair[i];
        mi[u] = x | dep_b;
        pi[u] = x | (uint64_t)dep_c;
        pp[u] = (V*)a.peer[b];
        va[u] = mine[mi[u]];
        vb[u] = pp[u][pi[u]];
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      const uint64_t w = w0 + (uint64_t)u * stride;
      if (w < total) {
        mine[mi[u]] = vb[u];
        pp[u][pi[u]] = va[u];
      }
    }
  }
}

class Circuit {
 public:
  explicit Circuit(int n) : n_(n), n_loc_(n) {}
  ~Circuit() { release(); }

  int n_;       // logical qubits
  int n_loc_;   // local physical positions (n_ - log2 world)
  int rank_ = 0, world_ = 1;
  qdc::ncclComm_t comm_ = nullptr;
  std::vector<Inst> insts_;
  cplx_t* state_ = nullptr;
  cplx_t* bwd_ = nullptr;
  cplx_t* initial_ = nullptr;  // nullptr <=> |0..0>
  cplx_t* stage_a_ = nullptr;  // exchange staging (half shard each; NCCL path only)
  cplx_t* stage_b_ = nullptr;
  // peer-memory exchange: partner buffers mapped with CUDA IPC
  static constexpr int kMaxWorld = 64;
  cplx_t* peer_state_[kMaxWorld] = {nullptr};
  cplx_t* peer_bwd_[kMaxWorld] = {nullptr};
  bool peer_ok_ = false;
  std::string peer_fail_;     // why the CUDA IPC mapping failed (reported by exchange() unless peer = 0)
  int opt_peer_ = 1;          // 1: peer-memory swap kernel when available, 0: NCCL send/recv + pack/unpack
  int* d_token_ = nullptr;    // 1 + kMaxWorld ints: tokens of the stream-ordered barriers (send slot, one receive slot per rank)
  int opt_multi_swap_ = 1;    // runs of remap swaps as ONE exchange with all ranks of the group (k_peer_multiswap)
  int opt_auto_swap_pos_ = 1; // sharded: lowest position of the remap victims chosen by the cost model (scheduler.hpp)
  int chosen_swap_min_pos_ = -1;
  Workspace ws_;
  double* d_res_ = nullptr;  // device results: 32 doubles per slot
  size_t d_res_slots_ = 0;
  std::vector<double> h_res_;
  // k-qubit densities: results (2 * 4^k doubles each, at kofs_[instruction]) and cotangents (4^k entries each,
  // at kmat_ofs_[instruction]) in regions of their own
  double* d_kres_ = nullptr;
  size_t d_kres_cap_ = 0;
  std::vector<double> h_kres_;
  std::vector<size_t> kofs_;
  cplx_t* d_kmat_ = nullptr;
  size_t d_kmat_cap_ = 0;
  std::vector<cplx_t> h_kmat_;
  std::vector<size_t> kmat_ofs_;
  // k-qubit gates, dense and diagonal: their device forms share the cotangents' region and copy (at
  // gmat_ofs_[instruction]); the gradients of the variable ones follow the 32-double slots in d_res_ (at
  // kgofs_[instruction], in doubles)
  std::vector<size_t> gmat_ofs_, kgofs_;
  cudaStream_t stream_ = 0;
  Stats stats_;
  int opt_fuse_ = 2;          // 0: one pass per instruction, 1: tiled multi-gate passes, 2: + register-blocked forward
  int opt_tile_strategy_ = 2;  // scheduler.hpp: 2 window growth with look-ahead, 1 window growth, 0 first-fit tiling
  int opt_batch_dens_ = 1;    // 1: densities / density seeds of one program point share tiled sweeps (tile_dens_kernels.cuh)
  int opt_soa_ = 1;           // f32 tile kernels: 1 pair-lane shared-memory layout (tile_soa_kernels.cuh), 0 interleaved
  // f32: 1 = windows of <= 6 qubits run as dense 64 x 64 blocks on the tensor cores (tc_exec.cuh / tc_block.cuh /
  // tc_rev.cuh); the scheduler then grows 6-position windows.  -1 (default): on for shards of >= 2^26 amplitudes,
  // where a block's sweep outweighs its host work (64 x 64 products, slice image, 96 KiB upload); 0: FP32-pipe tile
  // kernels only.
  int opt_tc_ = -1;
  int opt_tc_products_ = 6;   // bf16 slice products per block (tc_block.cuh): 6 = orders 0..2; 8 adds order 3 (2^-27 relative)
  int opt_tc_rev_ = 1;        // reverse step of a block: 1 one fused sweep (tc_rev.cuh, 4*S), 0 three sweeps (6*S)
  TcState* tc_ = nullptr;
  int opt_tile_bits_ = 0;  // 0: default for the precision
  int opt_low_bits_ = 0;
#ifdef QDC_F64
  int opt_max_tile_gates_ = 24;  // = QDC_TILE_MAXG_B, the capacity of the reverse kernel's parameter block
#else
  int opt_max_tile_gates_ = 32;
#endif
  Profiler prof_;
  qdc::Plan plan_;            // plan of the last forward sweep (backward replays it reversed)
  bool plan_all_dens_ = false;
  std::vector<int> exec_p2_, exec_p1_;  // physical positions each instruction ran at
  std::vector<int> cur_map_;            // logical qubit -> physical position of state_ right now (empty: identity)
  bool forward_valid_ = false;          // state_ holds the result of forward() of the CURRENT program

  void release() {
    if (state_) cudaFree(state_);
    if (bwd_) cudaFree(bwd_);
    if (initial_) cudaFree(initial_);
    if (stage_a_) cudaFree(stage_a_);
    if (stage_b_) cudaFree(stage_b_);
    if (d_res_) cudaFree(d_res_);
    if (d_kres_) cudaFree(d_kres_);
    if (d_kmat_) cudaFree(d_kmat_);
    state_ = bwd_ = initial_ = stage_a_ = stage_b_ = nullptr;
    d_res_ = nullptr;
    d_res_slots_ = 0;
    d_kres_ = nullptr;
    d_kmat_ = nullptr;
    d_kres_cap_ = d_kmat_cap_ = 0;
    ws_release(ws_);
    release_tiles();
#ifndef QDC_F64
    release_tc();
#endif
    for (int r = 0; r < kMaxWorld; r++) {
      if (peer_state_[r]) cudaIpcCloseMemHandle(peer_state_[r]);
      if (peer_bwd_[r]) cudaIpcCloseMemHandle(peer_bwd_[r]);
      peer_state_[r] = peer_bwd_[r] = nullptr;
    }
    if (d_token_) cudaFree(d_token_);
    d_token_ = nullptr;
    if (comm_) {
      qdc::nccl().CommDestroy(comm_);
      comm_ = nullptr;
    }
  }

  size_t bytes() const { return sizeof(cplx_t) << n_loc_; }

  const char* ensure_state() {
    if (!state_) QDC_CUDA(cudaMalloc((void**)&state_, bytes()));
    return nullptr;
  }

  // Sharding over `world` = 2^g ranks by the top g physical positions.
  const char* shard(int rank, int world, const void* unique_id) {
    if (world < 1 || (world & (world - 1)) != 0) return qdc_errf("world size must be a power of two.");
    int g = 0;
    while ((1 << g) < world) g++;
    if (g >= n_) return qdc_errf("more ranks than amplitudes.");
    // a dense two-qubit gate needs two local positions, and the exchange / streaming launchers split
    // the shard by vectors of 2^QDC_LV amplitudes
    if (world > 1 && n_ - g < 2 + QDC_LV)
      return qdc_errf("too many ranks: %d local qubits per rank, at least %d are needed.", n_ - g, 2 + QDC_LV);
    if (state_) QDC_CUDA(cudaFree(state_));
    state_ = nullptr;
    if (bwd_) QDC_CUDA(cudaFree(bwd_));
    bwd_ = nullptr;
    rank_ = rank;
    world_ = world;
    n_loc_ = n_ - g;
    if (world > 1) {
      const char* e = qdc::nccl().load();
      if (e) return qdc_errf("%s", e);
      qdc::ncclUniqueId id;
      memcpy(&id, unique_id, sizeof(id));
      const int rc = qdc::nccl().CommInitRank(&comm_, world, id, rank);
      if (rc != 0) return qdc_errf("ncclCommInitRank failed: %s", qdc::nccl().GetErrorString(rc));
    }
    QDC_TRY(ensure_state());
    if (world > 1) {
      QDC_CUDA(cudaMalloc((void**)&bwd_, bytes()));  // mapped by the partners: allocate up front
      QDC_CUDA(cudaMalloc((void**)&d_token_, (1 + kMaxWorld) * sizeof(int)));
      QDC_CUDA(cudaMemset(d_token_, 0, (1 + kMaxWorld) * sizeof(int)));
      setup_peers();
    }
    return nullptr;
  }

  // Map the partners' state / adjoint buffers (CUDA IPC).  Any failure just
  // leaves the NCCL send/recv path in charge.
  void setup_peers() {
    peer_ok_ = false;
    peer_fail_ = "the partner buffers could not be exchanged or mapped";
    if (world_ > kMaxWorld) {
      peer_fail_ = "world size above the peer table";
      return;
    }
    struct Handles { cudaIpcMemHandle_t s, b; };
    Handles mine;
    if (cudaIpcGetMemHandle(&mine.s, state_) != cudaSuccess || cudaIpcGetMemHandle(&mine.b, bwd_) != cudaSuccess) {
      peer_fail_ = std::string("cudaIpcGetMemHandle: ") + cudaGetErrorName(cudaGetLastError());
      return;
    }
    Handles *d_mine = nullptr, *d_all = nullptr;
    std::vector<Handles> all(world_);
    bool ok = cudaMalloc((void**)&d_mine, sizeof(Handles)) == cudaSuccess &&
              cudaMalloc((void**)&d_all, sizeof(Handles) * world_) == cudaSuccess;
    if (ok) ok = cudaMemcpy(d_mine, &mine, sizeof(Handles), cudaMemcpyHostToDevice) == cudaSuccess;
    if (ok) ok = qdc::nccl().AllGather(d_mine, d_all, sizeof(Handles), qdc::kNcclChar, comm_, stream_) == 0;
    if (ok) ok = cudaStreamSynchronize(stream_) == cudaSuccess;
    if (ok) ok = cudaMemcpy(all.data(), d_all, sizeof(Handles) * world_, cudaMemcpyDeviceToHost) == cudaSuccess;
    if (d_mine) cudaFree(d_mine);
    if (d_all) cudaFree(d_all);
    int mapped = ok ? 1 : 0;
    for (int p = 0; ok && p < world_; p++) {   // every rank: merged exchanges trade with all ranks of a group
      if (p == rank_) continue;
      void *ps = nullptr, *pb = nullptr;
      if (cudaIpcOpenMemHandle(&ps, all[p].s, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess ||
          cudaIpcOpenMemHandle(&pb, all[p].b, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        peer_fail_ = std::string("cudaIpcOpenMemHandle: ") + cudaGetErrorName(cudaGetLastError());
        mapped = 0;
        break;
      }
      peer_state_[p] = (cplx_t*)ps;
      peer_bwd_[p] = (cplx_t*)pb;
    }
    // every rank must take the same path: agree on success with an all-reduce (min via sum of failures)
    int* d_flag = nullptr;
    int fails = mapped ? 0 : 1, total = 1;
    if (cudaMalloc((void**)&d_flag, sizeof(int)) == cudaSuccess) {
      cudaMemcpy(d_flag, &fails, sizeof(int), cudaMemcpyHostToDevice);
      // int32 sum: ncclInt32 = 2
      if (qdc::nccl().AllReduce(d_flag, d_flag, 1, 2, qdc::kNcclSum, comm_, stream_) == 0 &&
          cudaStreamSynchronize(stream_) == cudaSuccess)
        cudaMemcpy(&total, d_flag, sizeof(int), cudaMemcpyDeviceToHost);
      cudaFree(d_flag);
    }
    peer_ok_ = (total == 0);
    if (peer_ok_) peer_fail_.clear();
    else if (mapped) peer_fail_ = "the mapping failed on another rank";
  }

  const char* ensure_results(size_t slots) {
    if (slots > d_res_slots_) {
      if (d_res_) QDC_CUDA(cudaFree(d_res_));
      QDC_CUDA(cudaMalloc((void**)&d_res_, slots * 32 * sizeof(double)));
      d_res_slots_ = slots;
    }
    h_res_.resize(slots * 32);
    return nullptr;
  }

  // In sharded mode `host` is this rank's shard (2^n_loc entries, identity qubit map).
  const char* set_state_from_host(const cplx_t* host, size_t len) {
    if (len == 0 || (len & (len - 1)) != 0) return qdc_errf("State size is not a power of 2.");
    if (len != ((size_t)1 << n_loc_))
      return qdc_errf("Size of the given state does not match the size of the tensor.");
    forward_valid_ = false;
    if (!initial_) QDC_CUDA(cudaMalloc((void**)&initial_, bytes()));
    QDC_CUDA(cudaMemcpy(initial_, host, bytes(), cudaMemcpyHostToDevice));
    return nullptr;
  }

  const char* add(int kind, size_t pos2, size_t pos1) {
    if (kind_is_k_dens(kind)) return qdc_errf("kind %d carries its qubits through qdc_circuit_add_dens.", kind);
    if (kind_is_k_gate(kind)) return qdc_errf("kind %d carries its qubits through qdc_circuit_add_gate.", kind);
    if (kind_is_diag_k(kind)) return qdc_errf("kind %d carries its qubits through qdc_circuit_add_gate_diag.", kind);
    if (kind < 0 || kind > K_DIFF_Q1_DENS) return qdc_errf("Unknown instruction kind %d.", kind);
    const bool one = kind_is_q1(kind) || kind_is_q1_dens(kind);
    if (one) {
      if (pos2 >= (size_t)n_) return qdc_errf("pos is out of the bound.");
    } else {
      if (pos1 == pos2) return qdc_errf("pos1 and pos2 must be different.");
      if (pos1 >= (size_t)n_) return qdc_errf("pos1 is out of the bound.");
      if (pos2 >= (size_t)n_) return qdc_errf("pos2 is out of the bound.");
    }
    insts_.push_back(Inst{kind, (int)pos2, one ? -1 : (int)pos1});
    forward_valid_ = false;
    return nullptr;
  }

  // Density on k = 1..6 qubits, positions[0] the most significant bit of its row and column index; k <= 2 adds the
  // one- and two-qubit kinds.
  const char* add_dens(const size_t* positions, size_t k, bool with_grad) {
    if (k < 1 || k > 6) return qdc_errf("the number of density qubits must be in 1..6, got %zu.", k);
    if (k == 1) return add(with_grad ? K_DIFF_Q1_DENS : K_Q1_DENS, positions[0], 0);
    if (k == 2) return add(with_grad ? K_DIFF_Q2_DENS : K_Q2_DENS, positions[0], positions[1]);
    Inst in{with_grad ? K_DIFF_DENS_K : K_DENS_K, -1, -1};
    for (size_t j = 0; j < k; j++) {
      if (positions[j] >= (size_t)n_) return qdc_errf("pos is out of the bound.");
      for (size_t i = 0; i < j; i++)
        if (positions[i] == positions[j]) return qdc_errf("positions must be different.");
      in.kpos[j] = (int)positions[j];
    }
    in.nk = (int)k;
    insts_.push_back(in);
    forward_valid_ = false;
    return nullptr;
  }

  // Gate on k = 1..6 qubits, positions[0] the most significant bit of its row and column index; k <= 2 adds the
  // one- and two-qubit kinds.
  const char* add_gate(const size_t* positions, size_t k, bool variable, bool non_unitary) {
    if (k < 1 || k > 6) return qdc_errf("the number of gate qubits must be in 1..6, got %zu.", k);
    if (k == 1)
      return add(variable ? (non_unitary ? K_VAR_Q1_NONU : K_VAR_Q1) : (non_unitary ? K_CONST_Q1_NONU : K_CONST_Q1),
                 positions[0], 0);
    if (k == 2)
      return add(variable ? (non_unitary ? K_VAR_Q2_NONU : K_VAR_Q2) : (non_unitary ? K_CONST_Q2_NONU : K_CONST_Q2),
                 positions[0], positions[1]);
    Inst in{variable ? (non_unitary ? K_VAR_GATE_K_NONU : K_VAR_GATE_K)
                     : (non_unitary ? K_CONST_GATE_K_NONU : K_CONST_GATE_K), -1, -1};
    for (size_t j = 0; j < k; j++) {
      if (positions[j] >= (size_t)n_) return qdc_errf("pos is out of the bound.");
      for (size_t i = 0; i < j; i++)
        if (positions[i] == positions[j]) return qdc_errf("positions must be different.");
      in.kpos[j] = (int)positions[j];
    }
    in.nk = (int)k;
    insts_.push_back(in);
    forward_valid_ = false;
    return nullptr;
  }

  // Diagonal gate on k = 1..6 qubits, positions[0] the most significant bit of its index j; a unitary one on
  // k = 2 adds the two-qubit diagonal kinds.
  const char* add_gate_diag(const size_t* positions, size_t k, bool variable, bool non_unitary) {
    if (k < 1 || k > 6) return qdc_errf("the number of gate qubits must be in 1..6, got %zu.", k);
    if (k == 2 && !non_unitary) return add(variable ? K_VAR_Q2_DIAG : K_CONST_Q2_DIAG, positions[0], positions[1]);
    Inst in{variable ? (non_unitary ? K_VAR_DIAG_K_NONU : K_VAR_DIAG_K)
                     : (non_unitary ? K_CONST_DIAG_K_NONU : K_CONST_DIAG_K), -1, -1};
    for (size_t j = 0; j < k; j++) {
      if (positions[j] >= (size_t)n_) return qdc_errf("pos is out of the bound.");
      for (size_t i = 0; i < j; i++)
        if (positions[i] == positions[j]) return qdc_errf("positions must be different.");
      in.kpos[j] = (int)positions[j];
    }
    in.nk = (int)k;
    insts_.push_back(in);
    forward_valid_ = false;
    return nullptr;
  }

  size_t count(int what) const {
    size_t c = 0;
    for (const Inst& in : insts_) {
      const int k = in.kind;
      const bool gate = kind_is_gate(k) || kind_is_k_gate(k) || kind_is_diag_k(k);
      switch (what) {
        case 0: c++; break;
        case 1: c += gate && !kind_is_var(k); break;
        case 2: c += gate && kind_is_var(k); break;
        case 3: c += kind_is_dens(k); break;
        case 4: c += kind_is_diff_dens(k); break;
        case 5: c += kind_is_dens(k) ? dens_len(in) : 0; break;
        case 6: c += kind_is_diff_dens(k) ? dens_len(in) : 0; break;
        case 7: c += (gate && kind_is_var(k)) ? gate_len(in) : 0; break;
      }
    }
    return c;
  }

  // Pair every gate instruction with its matrix (front-pop order of
  // src/circuit.rs:171-200, 222-251; equivalently the back-pop order of :278+).
  const char* bind_gates(const GateList& cg, const GateList& vg, std::vector<const cplx_t*>& ptr,
                         bool backward) {
    ptr.assign(insts_.size(), nullptr);
    size_t ci = 0, vi = 0, coff = 0, voff = 0;
    for (size_t i = 0; i < insts_.size(); i++) {
      const int k = insts_[i].kind;
      if (!kind_is_gate(k) && !kind_is_k_gate(k) && !kind_is_diag_k(k)) continue;
      const bool var = kind_is_var(k);
      const GateList& gl = var ? vg : cg;
      size_t& idx = var ? vi : ci;
      size_t& off = var ? voff : coff;
      if (idx >= gl.count) {
        if (backward) return qdc_errf("The number of gates is less than required.");
        return qdc_errf("The number of %s gates is less than required.", var ? "variable" : "constant");
      }
      if ((size_t)gl.lens[idx] != gate_len(insts_[i])) return qdc_errf("Incorrect len of the gate's buffer.");
      ptr[i] = gl.flat + off;
      off += gl.lens[idx];
      idx++;
    }
    if (ci != cg.count) return qdc_errf("Number of constant gates is more than required.");
    if (vi != vg.count)
      return qdc_errf(backward ? "Number of constant gates is more than required."
                               : "Number of variable gates is more than required.");
    return nullptr;
  }

  void account(uint64_t launches, uint64_t passes, uint64_t alg_passes) {
    stats_.kernel_launches += launches;
    stats_.hbm_passes += passes;
    stats_.algorithmic_bytes += alg_passes * (uint64_t)bytes();
  }

  const char* reset_state() {
    QDC_TRY(ensure_state());
    if (initial_) {
      QDC_TRY(eng_copy(stream_, initial_, state_, n_loc_));  // data_transfer, src/circuit.rs:174,225
    } else {
      QDC_CUDA(cudaMemsetAsync(state_, 0, bytes(), stream_));
      if (rank_ == 0) {
        k_set_one<<<1, 1, 0, stream_>>>(state_);
        QDC_CUDA(cudaGetLastError());
      }
      account(1, 0, 0);
    }
    return nullptr;
  }

  // ------------------------------------------------------- state I/O
  // Checkpoint format (SURVEY.md 8(f) item 4; the reference only has the
  // in-memory get_cpu_state_copy, src/quantized_tensor.rs:91-99): one file per
  // rank, 128-byte header + this rank's shard as raw little-endian interleaved
  // (re, im) pairs in PHYSICAL order (index bit p <-> physical position p).
  struct StateHeader {
    char magic[8];        // "QDCSTAT1"
    uint32_t real_bytes;  // 4 (f32) or 8 (f64)
    uint32_t n, n_loc, rank, world, reserved;
    uint8_t map[64];      // logical qubit q -> physical position (0xFF: unused); positions >= n_loc are rank bits
    uint8_t pad[32];
  };
  static_assert(sizeof(StateHeader) == 128, "header layout");
  static constexpr size_t kIoChunk = (size_t)32 << 20;

  const char* save_state(const char* path) {
    QDC_TRY(ensure_state());
    if (n_ > 64) return qdc_errf("state files hold at most 64 qubits.");
    StateHeader h;
    memset(&h, 0, sizeof(h));
    memcpy(h.magic, "QDCSTAT1", 8);
    h.real_bytes = (uint32_t)sizeof(real_t);
    h.n = (uint32_t)n_;
    h.n_loc = (uint32_t)n_loc_;
    h.rank = (uint32_t)rank_;
    h.world = (uint32_t)world_;
    memset(h.map, 0xFF, sizeof(h.map));
    for (int q = 0; q < n_; q++) h.map[q] = (uint8_t)(cur_map_.empty() ? q : cur_map_[q]);
    FILE* f = fopen(path, "wb");
    if (!f) return qdc_errf("cannot open %s for writing.", path);
    const char* err = nullptr;
    void* pin[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    auto fail = [&](const char* m) { if (!err) err = m; };
    if (fwrite(&h, sizeof(h), 1, f) != 1) fail(qdc_errf("short write to %s.", path));
    for (int k = 0; k < 2 && !err; k++) {
      if (cudaMallocHost(&pin[k], kIoChunk) != cudaSuccess || cudaEventCreate(&ev[k]) != cudaSuccess)
        fail(qdc_errf("cannot allocate the pinned staging buffers."));
    }
    // double-buffered: the D2H copy of chunk k+1 overlaps the fwrite of chunk k
    const size_t total = bytes(), nchunks = (total + kIoChunk - 1) / kIoChunk;
    auto issue = [&](size_t k) {
      const size_t off = k * kIoChunk, len = std::min(kIoChunk, total - off);
      if (cudaMemcpyAsync(pin[k & 1], (const char*)state_ + off, len, cudaMemcpyDeviceToHost, stream_) != cudaSuccess ||
          cudaEventRecord(ev[k & 1], stream_) != cudaSuccess)
        fail(qdc_errf("CUDA ERROR: device-to-host copy failed in save_state."));
    };
    if (!err && nchunks) issue(0);
    for (size_t k = 0; k < nchunks && !err; k++) {
      if (k + 1 < nchunks) issue(k + 1);
      if (err) break;
      if (cudaEventSynchronize(ev[k & 1]) != cudaSuccess) fail(qdc_errf("CUDA ERROR: save_state copy failed."));
      const size_t off = k * kIoChunk, len = std::min(kIoChunk, total - off);
      if (!err && fwrite(pin[k & 1], 1, len, f) != len) fail(qdc_errf("short write to %s.", path));
    }
    cudaStreamSynchronize(stream_);
    for (int k = 0; k < 2; k++) {
      if (pin[k]) cudaFreeHost(pin[k]);
      if (ev[k]) cudaEventDestroy(ev[k]);
    }
    if (fclose(f) != 0) fail(qdc_errf("cannot close %s.", path));
    return err;
  }

  // Load this rank's shard as the INITIAL state of the circuit (the role of
  // set_state_from_vector).  The file must be in the identity layout.
  const char* load_state(const char* path) {
    forward_valid_ = false;
    FILE* f = fopen(path, "rb");
    if (!f) return qdc_errf("cannot open %s for reading.", path);
    StateHeader h;
    const char* err = nullptr;
    auto fail = [&](const char* m) { if (!err) err = m; };
    if (fread(&h, sizeof(h), 1, f) != 1 || memcmp(h.magic, "QDCSTAT1", 8) != 0) fail(qdc_errf("%s is not a state file.", path));
    if (!err && h.real_bytes != sizeof(real_t))
      fail(qdc_errf("%s holds %u-byte reals, this build uses %zu-byte reals.", path, h.real_bytes, sizeof(real_t)));
    if (!err && ((int)h.n != n_ || (int)h.n_loc != n_loc_ || (int)h.rank != rank_ || (int)h.world != world_))
      fail(qdc_errf("%s is shard %u/%u of a %u-qubit state (%u local); this circuit is rank %d/%d of %d qubits (%d local).",
                    path, h.rank, h.world, h.n, h.n_loc, rank_, world_, n_, n_loc_));
    for (int q = 0; q < n_ && !err; q++)
      if (h.map[q] != q) fail(qdc_errf("%s is not in the identity qubit layout; re-save it after backward() or assemble it on the host.", path));
    void* pin[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    for (int k = 0; k < 2 && !err; k++) {
      if (cudaMallocHost(&pin[k], kIoChunk) != cudaSuccess || cudaEventCreate(&ev[k]) != cudaSuccess)
        fail(qdc_errf("cannot allocate the pinned staging buffers."));
    }
    if (!err && !initial_ && cudaMalloc((void**)&initial_, bytes()) != cudaSuccess) {
      initial_ = nullptr;
      fail(qdc_errf("CUDA ERROR: cannot allocate the initial-state buffer."));
    }
    const size_t total = bytes(), nchunks = (total + kIoChunk - 1) / kIoChunk;
    for (size_t k = 0; k < nchunks && !err; k++) {
      const size_t off = k * kIoChunk, len = std::min(kIoChunk, total - off);
      if (k >= 2 && cudaEventSynchronize(ev[k & 1]) != cudaSuccess) fail(qdc_errf("CUDA ERROR: load_state copy failed."));
      if (!err && fread(pin[k & 1], 1, len, f) != len) fail(qdc_errf("%s is truncated.", path));
      if (!err && (cudaMemcpyAsync((char*)initial_ + off, pin[k & 1], len, cudaMemcpyHostToDevice, stream_) != cudaSuccess ||
                   cudaEventRecord(ev[k & 1], stream_) != cudaSuccess))
        fail(qdc_errf("CUDA ERROR: host-to-device copy failed in load_state."));
    }
    if (cudaStreamSynchronize(stream_) != cudaSuccess) fail(qdc_errf("CUDA ERROR: load_state copy failed."));
    for (int k = 0; k < 2; k++) {
      if (pin[k]) cudaFreeHost(pin[k]);
      if (ev[k]) cudaEventDestroy(ev[k]);
    }
    fclose(f);
    return err;
  }

  // Current layout of the working state: out[q] = physical position of logical qubit q.
  void state_layout(int* out) const {
    for (int q = 0; q < n_; q++) out[q] = cur_map_.empty() ? q : cur_map_[q];
  }

  // ------------------------------------------------------------ planning
  static int sched_class(int k) {
    if (kind_is_q1(k)) return 0;
    if (kind_is_q2dense(k)) return 1;
    if (kind_is_diag(k)) return 2;
    if (kind_is_k_dens(k)) return 5;
    if (kind_is_k_gate(k)) return 6;
    if (kind_is_diag_k(k)) return 7;
    return kind_is_q1_dens(k) ? 3 : 4;
  }

  // One plan serves forward and backward; the backward kernel keeps state AND
  // adjoint tiles resident, so T is sized for it (2 * 2^T * sizeof(complex) = 64 KiB).
  int default_tile_bits() const {
#ifdef QDC_F64
    return 11;
#else
    return 12;
#endif
  }
  int min_tile_bits() const { return QDC_LV + 10; }
  int default_low_bits() const {
#ifdef QDC_F64
    return 3;
#else
    return 4;
#endif
  }

  bool tc_active() const {
#ifndef QDC_F64
    const bool on = opt_tc_ < 0 ? n_loc_ >= 26 : opt_tc_ != 0;
    return on && opt_fuse_ && n_loc_ >= 14;
#else
    return false;
#endif
  }

  // options of the gate scheduler: 6-position windows when the tensor-core blocks are on
  qdc::SchedOptions sched_options() const {
    qdc::SchedOptions so = base_options();
    if (tc_active() && so.tile_bits) {
      so.tile_bits = 6;
      so.low_bits = 0;
    }
    return so;
  }

  qdc::SchedOptions base_options() const {
    qdc::SchedOptions so;
    so.n = n_;
    so.n_loc = n_loc_;
    if (opt_fuse_) {
      so.tile_bits = opt_tile_bits_ ? opt_tile_bits_ : default_tile_bits();
      so.low_bits = opt_low_bits_ ? opt_low_bits_ : default_low_bits();
      so.max_tile_gates = opt_max_tile_gates_;
      so.tile_strategy = opt_tile_strategy_;
      if (so.tile_bits > n_loc_) so.tile_bits = n_loc_;
      if (so.tile_bits < min_tile_bits() || so.low_bits > so.tile_bits - 2) so.tile_bits = 0;  // too small to tile
    }
    return so;
  }

  // The plan depends only on the program (append-only), the density selection and the tunables: it is
  // rebuilt when one of them changed (scheduling the 1870-instruction test_autodiff circuit at 20 qubits
  // takes 2.7 ms, a quarter of its whole forward + backward).
  std::vector<long> plan_key_;
  void build_plan(bool all_dens) {
    const qdc::SchedOptions so = sched_options();
    const std::vector<long> key = {(long)insts_.size(), all_dens ? 1L : 0L, so.n, so.n_loc, so.tile_bits, so.low_bits,
                                   so.max_tile_gates, so.min_tile_gates, so.group_bits, so.swap_min_pos, so.tile_strategy,
                                   tc_active() ? 1L : 0L, (long)opt_auto_swap_pos_,
                                   (peer_ok_ && opt_peer_ && opt_multi_swap_) ? 1L : 0L};
    if (key == plan_key_ && !plan_.steps.empty()) return;
    plan_key_ = key;
    std::vector<qdc::SchedInst> si(insts_.size());
    for (size_t i = 0; i < insts_.size(); i++) {
      const int k = insts_[i].kind;
      si[i].kind_class = sched_class(k);
      si[i].q2 = insts_[i].pos2;
      si[i].q1 = insts_[i].pos1;
      si[i].skip = kind_is_dens(k) && !all_dens && !kind_is_diff_dens(k);
      si[i].nq = insts_[i].nk;
      for (int j = 0; j < insts_[i].nk; j++) si[i].qk[j] = insts_[i].kpos[j];
    }
    if (world_ > 1 && opt_auto_swap_pos_) {
      // sharded: where the remap victims may sit is decided by the cost model of scheduler.hpp (every rank builds the
      // same plan: the choice is a pure function of the program and the options)
      qdc::CostModel cm;
      cm.amp_bytes = (int)sizeof(cplx_t);
      cm.vec_log2 = QDC_LV;
      cm.merged = peer_ok_ && opt_peer_ && opt_multi_swap_;
#ifdef QDC_F64
      cm.tile_ms = 640;
      cm.gate_ms = 70;
      cm.shard_ms = 98.8;
#else
      cm.tile_ms = tc_active() ? 59 : 280;
#endif
      plan_ = qdc::schedule_best(si, so, cm, &chosen_swap_min_pos_);
    } else {
      qdc::Scheduler sch(si, so);
      plan_ = sch.run();
      chosen_swap_min_pos_ = so.swap_min_pos;
    }
    plan_all_dens_ = all_dens;
    exec_p2_.assign(insts_.size(), -1);
    exec_p1_.assign(insts_.size(), -1);
    diag_hilo_.assign(insts_.size(), 0);
    auto note = [&](const qdc::Step& st) {
      if (st.inst >= 0) {
        exec_p2_[st.inst] = st.p2;
        exec_p1_[st.inst] = st.p1;
      }
    };
    for (const qdc::Step& st : plan_.steps) note(st);
    for (const qdc::Step& st : plan_.tile_steps) note(st);
  }

  // ------------------------------------------------- diagonal on global bits
  // Effective local form of a diagonal gate some of whose positions are rank
  // bits: returns the 4 entries to feed the elementwise kernel selected by
  // (sel2, sel1) (both local).  j' = 2 bit(sel2) + bit(sel1) takes only the
  // values 0 and 3 when sel2 == sel1.
  void effective_diag(const cplx_t* d, int p2, int p1, cplx_t (&e)[4], int& sel2, int& sel1) const {
    const bool g2 = p2 >= n_loc_, g1 = p1 >= n_loc_;
    const int c2 = g2 ? (rank_ >> (p2 - n_loc_)) & 1 : 0, c1 = g1 ? (rank_ >> (p1 - n_loc_)) & 1 : 0;
    for (int j = 0; j < 4; j++) e[j] = d[j];
    sel2 = p2;
    sel1 = p1;
    if (g2 && g1) {
      e[0] = e[3] = d[2 * c2 + c1];
      sel2 = sel1 = 0;
    } else if (g2) {
      e[0] = d[2 * c2 + 0];
      e[3] = d[2 * c2 + 1];
      sel2 = sel1 = p1;
    } else if (g1) {
      e[0] = d[0 + c1];
      e[3] = d[2 + c1];
      sel2 = sel1 = p2;
    }
  }

  // kernel-order diagonal gradient (8 doubles) -> reference order on this rank
  void scatter_diag_grad(const double* h, int p2, int p1, zc (&out)[4]) const {
    const bool g2 = p2 >= n_loc_, g1 = p1 >= n_loc_;
    const int c2 = g2 ? (rank_ >> (p2 - n_loc_)) & 1 : 0, c1 = g1 ? (rank_ >> (p1 - n_loc_)) & 1 : 0;
    for (int j = 0; j < 4; j++) out[j] = zc(0, 0);
    if (!g2 && !g1) {
      for (int j = 0; j < 4; j++) out[j] = zc(h[2 * j], h[2 * j + 1]);
    } else if (g2 && g1) {
      out[2 * c2 + c1] = zc(h[0] + h[6], h[1] + h[7]);
    } else if (g2) {
      out[2 * c2 + 0] = zc(h[0], h[1]);
      out[2 * c2 + 1] = zc(h[6], h[7]);
    } else {
      out[0 + c1] = zc(h[0], h[1]);
      out[2 + c1] = zc(h[6], h[7]);
    }
  }

  // ---------------------------------------------------------- exchanges
  const char* ensure_staging() {
    const size_t half = bytes() / 2;
    if (!stage_a_) QDC_CUDA(cudaMalloc((void**)&stage_a_, half));
    if (!stage_b_) QDC_CUDA(cudaMalloc((void**)&stage_b_, half));
    return nullptr;
  }

  template <bool GATHER>
  const char* half_copy(cplx_t* full, cplx_t* half, int pos, int val) {
    DeviceInfo di;
    QDC_TRY(qdc_device_info(&di));
    if (pos >= QDC_LV) {
      const uint64_t nhalf = 1ull << (n_loc_ - 1 - QDC_LV);
      const int grid = pick_grid(nhalf, 1, 8, di.sm_count);
      k_half_copy<vec_t, GATHER><<<grid, QDC_BLOCK, 0, stream_>>>((vec_t*)full, (vec_t*)half, pos - QDC_LV, val,
                                                                  nhalf);
    } else {
      const uint64_t nhalf = 1ull << (n_loc_ - 1);
      const int grid = pick_grid(nhalf, 1, 8, di.sm_count);
      k_half_copy<cplx_t, GATHER><<<grid, QDC_BLOCK, 0, stream_>>>(full, half, pos, val, nhalf);
    }
    QDC_CUDA(cudaGetLastError());
    return nullptr;
  }

  // Swap global bit `gbit` with local position `lpos` of buffer `buf`:
  // new[lpos=b, rank bit=c] = old[lpos=c, rank bit=b].  This rank keeps its
  // half lpos == c and trades its half lpos == 1-c for the partner's half
  // lpos == c (the partner sees the mirror image).
  // Stream-ordered rendezvous with one partner: returns (on the stream) only
  // after the partner's stream has reached the matching call.
  const char* pair_barrier(int partner) {
    qdc::NcclApi& api = qdc::nccl();
    int rc = api.GroupStart();
    if (rc == 0) rc = api.Send(d_token_, sizeof(int), qdc::kNcclChar, partner, comm_, stream_);
    if (rc == 0) rc = api.Recv(d_token_ + 1, sizeof(int), qdc::kNcclChar, partner, comm_, stream_);
    const int rc2 = api.GroupEnd();
    if (rc == 0) rc = rc2;
    if (rc != 0) return qdc_errf("NCCL barrier failed: %s", api.GetErrorString(rc));
    return nullptr;
  }

  const char* exchange_peer(cplx_t* buf, int gbit, int lpos) {
    const int c = (rank_ >> gbit) & 1, partner = rank_ ^ (1 << gbit);
    cplx_t* peer = (buf == state_) ? peer_state_[partner] : peer_bwd_[partner];
    DeviceInfo di;
    QDC_TRY(qdc_device_info(&di));
    QDC_TRY(pair_barrier(partner));  // both GPUs are done with everything before the swap
    if (lpos >= QDC_LV) {
      const uint64_t nhalf = 1ull << (n_loc_ - 1 - QDC_LV);
      const uint64_t lo = c ? nhalf / 2 : 0, hi = c ? nhalf : nhalf / 2;
      const int grid = pick_grid(hi - lo, 4, 8, di.sm_count);
      k_peer_swap<vec_t><<<grid, QDC_BLOCK, 0, stream_>>>((vec_t*)buf, (vec_t*)peer, lpos - QDC_LV, c, lo, hi);
    } else {
      const uint64_t nhalf = 1ull << (n_loc_ - 1);
      const uint64_t lo = c ? nhalf / 2 : 0, hi = c ? nhalf : nhalf / 2;
      const int grid = pick_grid(hi - lo, 4, 8, di.sm_count);
      k_peer_swap<cplx_t><<<grid, QDC_BLOCK, 0, stream_>>>(buf, peer, lpos, c, lo, hi);
    }
    QDC_CUDA(cudaGetLastError());
    QDC_TRY(pair_barrier(partner));  // the partner's half of the pairs has landed here too
    account(1, 1, 0);
    return nullptr;
  }

  // Stream-ordered rendezvous with several partners at once (one NCCL group).
  const char* group_barrier(const int* partners, int count) {
    qdc::NcclApi& api = qdc::nccl();
    int rc = api.GroupStart();
    for (int i = 0; i < count && rc == 0; i++) {
      rc = api.Send(d_token_, sizeof(int), qdc::kNcclChar, partners[i], comm_, stream_);
      if (rc == 0) rc = api.Recv(d_token_ + 1 + partners[i], sizeof(int), qdc::kNcclChar, partners[i], comm_, stream_);
    }
    const int rc2 = api.GroupEnd();
    if (rc == 0) rc = rc2;
    if (rc != 0) return qdc_errf("NCCL barrier failed: %s", api.GetErrorString(rc));
    return nullptr;
  }

  // Can the swaps (gbit[i] <-> lpos[i]), i < k, run as one merged exchange?
  bool multi_swap_ok(int k, const int* lpos) const {
    if (!(peer_ok_ && opt_peer_ && opt_multi_swap_) || k < 2 || k > 3) return false;
    for (int i = 0; i < k; i++)
      if (lpos[i] < QDC_LV) return false;
    return n_loc_ - QDC_LV - k - 1 >= 0;
  }

  // k simultaneous swaps gbit[i] <-> lpos[i] of buffer `buf` (k_peer_multiswap)
  const char* exchange_multi(cplx_t* buf, int k, const int* gbit, const int* lpos) {
    MultiSwapArgs a;
    a.k = k;
    a.c = 0;
    for (int i = 0; i < k; i++) {
      a.c |= ((rank_ >> gbit[i]) & 1) << i;
      a.pos_pair[i] = lpos[i] - QDC_LV;
      a.pos_sorted[i] = lpos[i] - QDC_LV;
    }
    std::sort(a.pos_sorted, a.pos_sorted + k);
    a.half_log2 = n_loc_ - QDC_LV - k - 1;
    int partners[8], np = 0;
    for (int b = 0; b < (1 << k); b++) {
      a.peer[b] = nullptr;
      if (b == a.c) continue;
      int p = rank_;
      for (int i = 0; i < k; i++) p = (p & ~(1 << gbit[i])) | (((b >> i) & 1) << gbit[i]);
      a.peer[b] = (buf == state_) ? (void*)peer_state_[p] : (void*)peer_bwd_[p];
      if (!a.peer[b]) return qdc_errf("internal: rank %d is not mapped for the merged exchange.", p);
      partners[np++] = p;
    }
    DeviceInfo di;
    QDC_TRY(qdc_device_info(&di));
    QDC_TRY(group_barrier(partners, np));   // every rank of the group is done with everything before the exchange
    const uint64_t total = (uint64_t)((1 << k) - 1) << a.half_log2;
    const int grid = pick_grid(total, 4, 8, di.sm_count);
    k_peer_multiswap<vec_t><<<grid, QDC_BLOCK, 0, stream_>>>((vec_t*)buf, a);
    QDC_CUDA(cudaGetLastError());
    QDC_TRY(group_barrier(partners, np));   // the partners' halves of the pairs have landed here too
    account(1, 1, 0);
    return nullptr;
  }

  // The run of consecutive SWAP steps starting at plan step `si` (walking by `dir` = +1 / -1) that can be merged:
  // returns how many (1 = no merge) and their (gbit, lpos).
  int swap_run(size_t si, int dir, int* gbit, int* lpos) const {
    const std::vector<qdc::Step>& steps = plan_.steps;
    int k = 0;
    for (size_t j = si; j < steps.size() && k < 3; j += (size_t)dir) {   // (j wraps past 0 to SIZE_MAX: loop ends)
      const qdc::Step& t = steps[j];
      if (t.type != qdc::ST_SWAP) break;
      bool clash = false;
      for (int i = 0; i < k; i++) clash |= gbit[i] == t.gbit || lpos[i] == t.lpos;
      if (clash) break;
      gbit[k] = t.gbit;
      lpos[k] = t.lpos;
      k++;
    }
    if (k >= 2 && !multi_swap_ok(k, lpos)) return 1;
    return k;
  }

  const char* exchange(cplx_t* buf, int gbit, int lpos) {
    if (peer_ok_ && opt_peer_) return exchange_peer(buf, gbit, lpos);
    // No silent performance cliff (the NCCL path runs at ~2/3 of the peer kernel's rate and needs 2 x half a
    // shard of staging): falling back is the caller's decision, option peer = 0.
    if (opt_peer_)
      return qdc_errf("peer-memory exchange unavailable (%s); set option \"peer\" to 0 for the NCCL send/recv exchange.",
                      peer_fail_.c_str());
    QDC_TRY(ensure_staging());
    const int c = (rank_ >> gbit) & 1, partner = rank_ ^ (1 << gbit);
    const size_t half_bytes = bytes() / 2;
    const bool top = lpos == n_loc_ - 1;
    cplx_t* out_half = top ? buf + ((size_t)(1 - c) << (n_loc_ - 1)) : stage_a_;
    if (!top) QDC_TRY((half_copy<true>(buf, stage_a_, lpos, 1 - c)));
    qdc::NcclApi& api = qdc::nccl();
    int rc = api.GroupStart();
    if (rc == 0) rc = api.Send(out_half, half_bytes, qdc::kNcclChar, partner, comm_, stream_);
    if (rc == 0) rc = api.Recv(stage_b_, half_bytes, qdc::kNcclChar, partner, comm_, stream_);
    const int rc2 = api.GroupEnd();
    if (rc == 0) rc = rc2;
    if (rc != 0) return qdc_errf("NCCL exchange failed: %s", api.GetErrorString(rc));
    if (top) {
      QDC_CUDA(cudaMemcpyAsync(out_half, stage_b_, half_bytes, cudaMemcpyDeviceToDevice, stream_));
    } else {
      QDC_TRY((half_copy<false>(buf, stage_b_, lpos, 1 - c)));
    }
    account(top ? 1 : 2, 1, 0);
    return nullptr;
  }

  // ------------------------------------------------------------- forward
  const char* sweep(const GateList& cg, const GateList& vg, bool all_dens, cplx_t* out, size_t cap,
                    size_t* out_len) {
    if (insts_.empty()) return qdc_errf("The circuit is empty.");
    stats_ = Stats();
    prof_.reset();
    std::vector<const cplx_t*> gp;
    QDC_TRY(bind_gates(cg, vg, gp, false));
    const size_t need = count(all_dens ? 5 : 6);
    if (cap < need) return qdc_errf("Output buffer too small: %zu < %zu.", cap, need);
    // 32-double slots of the one- and two-qubit densities; offsets of the k-qubit ones in their own region
    size_t nslots = 0, nkres = 0;
    kofs_.assign(insts_.size(), 0);
    for (size_t i = 0; i < insts_.size(); i++) {
      const Inst& in = insts_[i];
      if (!kind_is_dens(in.kind) || (!all_dens && !kind_is_diff_dens(in.kind))) continue;
      if (!kind_is_k_dens(in.kind)) {
        nslots++;
        continue;
      }
      kofs_[i] = nkres;
      nkres += 2 * dens_len(in);
    }
    QDC_TRY(ensure_results(nslots));
    if (nkres > d_kres_cap_) {
      if (d_kres_) QDC_CUDA(cudaFree(d_kres_));
      d_kres_ = nullptr;
      QDC_CUDA(cudaMalloc((void**)&d_kres_, nkres * sizeof(double)));
      d_kres_cap_ = nkres;
    }
    h_kres_.resize(nkres);
    forward_valid_ = false;
    build_plan(all_dens);   // (the diagonal k-qubit gates' forms depend on where the plan runs them)
    if (!plan_.ok)
      return qdc_errf("the program cannot be scheduled on %d local qubits per rank (an instruction never has all "
                      "its qubits local).", n_loc_);
    h_kmat_.clear();
    QDC_TRY(add_gate_k_forms(gp, false));
    QDC_TRY(upload_kmat());
    QDC_TRY(reset_state());
    if (nslots) QDC_CUDA(cudaMemsetAsync(d_res_, 0, nslots * 32 * sizeof(double), stream_));
#ifndef QDC_F64
    QDC_TRY(tc_begin(false));
#endif
    QDC_TRY(run_forward(gp, all_dens));
    cur_map_ = plan_.final_map;
    forward_valid_ = true;
    // single read-back of every density
    if (nslots) {
      QDC_CUDA(cudaMemcpyAsync(h_res_.data(), d_res_, nslots * 32 * sizeof(double), cudaMemcpyDeviceToHost,
                               stream_));
    }
    if (nkres)
      QDC_CUDA(cudaMemcpyAsync(h_kres_.data(), d_kres_, nkres * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    QDC_CUDA(cudaStreamSynchronize(stream_));
    if (prof_.on) prof_.collect();
    size_t slot = 0, o = 0;
    for (size_t i = 0; i < insts_.size(); i++) {
      const Inst& in = insts_[i];
      if (!kind_is_dens(in.kind)) continue;
      if (!all_dens && !kind_is_diff_dens(in.kind)) continue;
      if (kind_is_k_dens(in.kind)) {
        const size_t len = dens_len(in);
        const double* h = &h_kres_[kofs_[i]];
        for (size_t j = 0; j < len; j++) {
          out[o + j].x = (real_t)h[2 * j];
          out[o + j].y = (real_t)h[2 * j + 1];
        }
        o += len;
        continue;
      }
      const double* h = &h_res_[slot * 32];
      if (kind_is_q1_dens(in.kind)) {
        for (int j = 0; j < 4; j++) {
          out[o + j].x = (real_t)h[2 * j];
          out[o + j].y = (real_t)h[2 * j + 1];
        }
        o += 4;
      } else {
        zc m[16];
        unpermute_q2(h, exec_p2_[i] < exec_p1_[i], m);
        for (int j = 0; j < 16; j++) {
          out[o + j].x = (real_t)m[j].real();
          out[o + j].y = (real_t)m[j].imag();
        }
        o += 16;
      }
      slot++;
    }
    *out_len = o;
    return nullptr;
  }

  const char* fwd_gate_step(const qdc::Step& st, const std::vector<const cplx_t*>& gp) {
    const int k = insts_[st.inst].kind;
    if (kind_is_q1(k)) {
      PROF(CAT_FWD_Q1, 2, eng_q1gate(stream_, ws_, state_, gp[st.inst], FORM_PLAIN, st.p2, n_loc_));
    } else if (kind_is_q2dense(k)) {
      PROF(CAT_FWD_Q2, 2, eng_q2gate(stream_, ws_, state_, gp[st.inst], FORM_PLAIN, st.p2, st.p1, n_loc_));
    } else {
      cplx_t e[4];
      int s2, s1;
      effective_diag(gp[st.inst], st.p2, st.p1, e, s2, s1);
      PROF(CAT_FWD_DIAG, 2, eng_q2diag(stream_, ws_, state_, e, false, s2, s1, n_loc_));
    }
    account(1, 1, 2);
    return nullptr;
  }

  const char* run_forward(const std::vector<const cplx_t*>& gp, bool all_dens) {
    // output slot of every evaluated density, in program order
    std::vector<long> dslot(insts_.size(), -1);
    {
      long s = 0;
      for (size_t i = 0; i < insts_.size(); i++) {
        const int k = insts_[i].kind;
        if (kind_is_dens(k) && !kind_is_k_dens(k) && (all_dens || kind_is_diff_dens(k))) dslot[i] = s++;
      }
    }
    const std::vector<qdc::Step>& steps = plan_.steps;
    for (size_t si = 0; si < steps.size(); si++) {
      const qdc::Step& st = steps[si];
      switch (st.type) {
        case qdc::ST_GATE:
          QDC_TRY(fwd_gate_step(st, gp));
          break;
        case qdc::ST_TILE:
#ifndef QDC_F64
          if (tc_step_ok(st)) {
            QDC_TRY(run_tc_forward(st, gp, false));
            break;
          }
#endif
          if (opt_fuse_ >= 2) QDC_TRY(run_tile_forward_blocked(st, gp, false));
          else QDC_TRY(run_tile_forward(st, gp));
          break;
        case qdc::ST_SWAP: {
          int gb[3], lp[3];
          const int k = swap_run(si, +1, gb, lp);
          if (k >= 2) {
            PROF(CAT_EXCHANGE, 0, exchange_multi(state_, k, gb, lp));
            si += (size_t)(k - 1);
          } else {
            PROF(CAT_EXCHANGE, 0, exchange(state_, st.gbit, st.lpos));
          }
          break;
        }
        case qdc::ST_DENS: {
          size_t sj = si;  // the run of densities requested at this program point
          while (sj + 1 < steps.size() && steps[sj + 1].type == qdc::ST_DENS) sj++;
          QDC_TRY(run_dens_run(si, sj, dslot));
          si = sj;
          break;
        }
        case qdc::ST_GATE_K:
          QDC_TRY(gate_k_apply(st, state_, d_kmat_ + gmat_ofs_[st.inst], CAT_GATE_K_FWD));
          break;
        case qdc::ST_DIAG_K:
          QDC_TRY(diag_k_apply(st, state_, d_kmat_ + gmat_ofs_[st.inst], CAT_DIAG_K_FWD));
          break;
      }
    }
    return nullptr;
  }

  const char* dens_single(const qdc::Step& st, const std::vector<long>& dslot) {
    double* dst = d_res_ + (size_t)dslot[st.inst] * 32;
    if (st.p1 < 0) {
      PROF(CAT_DENSITY, 1, eng_dens_q1(stream_, ws_, state_, st.p2, n_loc_, dst));
    } else {
      PROF(CAT_DENSITY, 1, eng_dens_q2(stream_, ws_, state_, st.p2, st.p1, n_loc_, dst));
    }
    account(2, 1, 1);
    return nullptr;
  }

  const char* seed_single(const qdc::Step& st, const std::vector<const cplx_t*>& dp, bool live) {
    if (st.p1 < 0) {
      PROF(CAT_SEED, live ? 3 : 2, eng_seed_q1(stream_, ws_, state_, bwd_, dp[st.inst], st.p2, n_loc_, live));
    } else {
      PROF(CAT_SEED, live ? 3 : 2,
           eng_seed_q2(stream_, ws_, state_, bwd_, dp[st.inst], st.p2, st.p1, n_loc_, live));
    }
    account(1, 1, live ? 3 : 2);
    return nullptr;
  }

  // Appends the device forms of every k-qubit gate (gate_k_forms, diag_k_forms) to h_kmat_, at
  // gmat_ofs_[instruction].
  const char* add_gate_k_forms(const std::vector<const cplx_t*>& gp, bool reverse) {
    gmat_ofs_.assign(insts_.size(), 0);
    for (size_t i = 0; i < insts_.size(); i++) {
      const Inst& in = insts_[i];
      if (!kind_is_k_gate(in.kind)) continue;
      gmat_ofs_[i] = h_kmat_.size();
      QDC_TRY(gate_k_forms(gp[i], in.nk, kind_is_nonu(in.kind), reverse, &h_kmat_));
    }
    for (const qdc::Step& st : plan_.steps) {   // diagonal ones: folded over the rank bits of their plan step
      if (st.type != qdc::ST_DIAG_K) continue;
      gmat_ofs_[st.inst] = h_kmat_.size();
      QDC_TRY(diag_k_forms(gp[st.inst], insts_[st.inst], st.pk, reverse, &h_kmat_));
    }
    return nullptr;
  }

  // h_kmat_ -> d_kmat_, one copy per call
  const char* upload_kmat() {
    if (h_kmat_.empty()) return nullptr;
    if (h_kmat_.size() > d_kmat_cap_) {
      if (d_kmat_) QDC_CUDA(cudaFree(d_kmat_));
      d_kmat_ = nullptr;
      QDC_CUDA(cudaMalloc((void**)&d_kmat_, h_kmat_.size() * sizeof(cplx_t)));
      d_kmat_cap_ = h_kmat_.size();
    }
    QDC_CUDA(cudaMemcpyAsync(d_kmat_, h_kmat_.data(), h_kmat_.size() * sizeof(cplx_t), cudaMemcpyHostToDevice,
                             stream_));
    return nullptr;
  }

  // ------------------------------------------------------------ backward
  const char* backward(const GateList& dg, const GateList& cg, const GateList& vg, cplx_t* out, size_t cap,
                       size_t* out_len) {
    if (insts_.empty()) return qdc_errf("The circuit is empty.");
    // The reverse pass un-computes the state forward() left behind, replaying ITS plan: valid once per
    // forward() of the unchanged program (src/circuit.rs:266-429 consumes self.state the same way).
    if (!state_ || plan_.steps.empty() || !forward_valid_ || plan_key_.empty() || plan_key_[0] != (long)insts_.size())
      return qdc_errf("backward() must follow a forward() of the same program (once per forward).");
    forward_valid_ = false;
    stats_ = Stats();
    prof_.reset();
    std::vector<const cplx_t*> gp;
    QDC_TRY(bind_gates(cg, vg, gp, true));
    // cotangents: one per Diff* density, program order
    std::vector<const cplx_t*> dp(insts_.size(), nullptr);
    {
      size_t di = 0, off = 0;
      for (size_t i = 0; i < insts_.size(); i++) {
        if (!kind_is_diff_dens(insts_[i].kind)) continue;
        if (di >= dg.count)
          return qdc_errf("The number of gradients wrt density matrices is less than required.");
        if ((size_t)dg.lens[di] != dens_len(insts_[i]))
          return qdc_errf("Incorrect len of the gate's buffer.");
        dp[i] = dg.flat + off;
        off += dg.lens[di];
        di++;
      }
      if (di != dg.count) return qdc_errf("Number of gradients wrt density matrices is more than required.");
    }
    // cotangents of the k-qubit densities go to the device in one copy (their seeds read them from there)
    kmat_ofs_.assign(insts_.size(), 0);
    h_kmat_.clear();
    for (size_t i = 0; i < insts_.size(); i++) {
      if (insts_[i].kind != K_DIFF_DENS_K) continue;
      kmat_ofs_[i] = h_kmat_.size();
      h_kmat_.insert(h_kmat_.end(), dp[i], dp[i] + dens_len(insts_[i]));
    }
    QDC_TRY(add_gate_k_forms(gp, true));
    const size_t need = count(7);
    if (cap < need) return qdc_errf("Output buffer too small: %zu < %zu.", cap, need);
    // variable-gate slot of every one- and two-qubit instruction
    std::vector<long> vslot(insts_.size(), -1);
    {
      long s = 0;
      for (size_t i = 0; i < insts_.size(); i++)
        if (kind_is_gate(insts_[i].kind) && kind_is_var(insts_[i].kind)) vslot[i] = s++;
    }
    const size_t nvar = (size_t)std::count_if(vslot.begin(), vslot.end(), [](long s) { return s >= 0; });
    // gradients of the variable k-qubit gates: 2 * 4^k doubles each, after the slots
    size_t ndbl = nvar * 32;
    kgofs_.assign(insts_.size(), 0);
    for (size_t i = 0; i < insts_.size(); i++) {
      if (!(kind_is_k_gate(insts_[i].kind) || kind_is_diag_k(insts_[i].kind)) || !kind_is_var(insts_[i].kind)) continue;
      kgofs_[i] = ndbl;
      ndbl += 2 * gate_len(insts_[i]);
    }
    QDC_TRY(ensure_results((ndbl + 31) / 32));
    if (ndbl) QDC_CUDA(cudaMemsetAsync(d_res_, 0, ndbl * sizeof(double), stream_));
    if (!bwd_) QDC_CUDA(cudaMalloc((void**)&bwd_, bytes()));  // (sharded mode allocated it in shard())
    QDC_TRY(upload_kmat());
#ifndef QDC_F64
    QDC_TRY(tc_begin(true));
#endif
    QDC_TRY(run_backward(gp, dp, vslot));
    cur_map_.clear();  // every swap has been replayed in reverse: identity layout again
    if (ndbl)
      QDC_CUDA(cudaMemcpyAsync(h_res_.data(), d_res_, ndbl * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    QDC_CUDA(cudaStreamSynchronize(stream_));
    if (prof_.on) prof_.collect();
#ifndef QDC_F64
    QDC_TRY(tc_finish_backward());
#endif
    size_t o = 0;
    for (size_t i = 0; i < insts_.size(); i++) {
      const Inst& in = insts_[i];
      if (kind_is_k_gate(in.kind) && kind_is_var(in.kind)) {
        const size_t len = gate_len(in);
        const double* h = &h_res_[kgofs_[i]];
        for (size_t j = 0; j < len; j++) {
          out[o + j].x = (real_t)h[2 * j];
          out[o + j].y = (real_t)h[2 * j + 1];
        }
        o += len;
        continue;
      }
      if (kind_is_diag_k(in.kind) && kind_is_var(in.kind)) {
        // the kernel's 2^k_loc entries -> the gate's 2^k entries at this rank's bits
        std::vector<zc> g;
        qdc::diag_scatter(qdc::diag_fold_split(exec_pk(i), in.nk, n_loc_, rank_), in.nk, &h_res_[kgofs_[i]], &g);
        for (size_t j = 0; j < g.size(); j++) {
          out[o + j].x = (real_t)g[j].real();
          out[o + j].y = (real_t)g[j].imag();
        }
        o += g.size();
        continue;
      }
      if (vslot[i] < 0) continue;
#ifndef QDC_F64
      if (const std::vector<zc>* tg = tc_gradient(i)) {   // gate of a tensor-core block: already in reference order
        for (size_t j = 0; j < tg->size(); j++) {
          out[o + j].x = (real_t)(*tg)[j].real();
          out[o + j].y = (real_t)(*tg)[j].imag();
        }
        o += tg->size();
        continue;
      }
#endif
      const double* h = &h_res_[(size_t)vslot[i] * 32];
      if (kind_is_q2dense(in.kind)) {
        zc m[16];
        unpermute_q2(h, exec_p2_[i] < exec_p1_[i], m);
        for (int j = 0; j < 16; j++) {
          out[o + j].x = (real_t)m[j].real();
          out[o + j].y = (real_t)m[j].imag();
        }
        o += 16;
      } else if (kind_is_diag(in.kind)) {
        zc m[4];
        scatter_diag_grad(h, exec_p2_[i], exec_p1_[i], m);
        if (diag_hilo_[i]) std::swap(m[1], m[2]);
        for (int j = 0; j < 4; j++) {
          out[o + j].x = (real_t)m[j].real();
          out[o + j].y = (real_t)m[j].imag();
        }
        o += 4;
      } else {
        for (int j = 0; j < 4; j++) {
          out[o + j].x = (real_t)h[2 * j];
          out[o + j].y = (real_t)h[2 * j + 1];
        }
        o += 4;
      }
    }
    *out_len = o;
    return nullptr;
  }

  const char* bwd_gate_step(const qdc::Step& st, const std::vector<const cplx_t*>& gp,
                            const std::vector<long>& vslot, bool live) {
    const int ii = st.inst;
    const int k = insts_[ii].kind;
    const int inv_form = kind_is_nonu(k) ? FORM_INV : FORM_CONJ_TR;
    double* gdst = (vslot[ii] >= 0) ? d_res_ + (size_t)vslot[ii] * 32 : nullptr;
    cplx_t e[4];
    int s2 = st.p2, s1 = st.p1;
    if (kind_is_diag(k)) effective_diag(gp[ii], st.p2, st.p1, e, s2, s1);
    if (!live) {
      // no adjoint yet: un-compute only; variable gates keep their zero gradient
      if (kind_is_q1(k)) {
        PROF(CAT_UNCOMPUTE, 2, eng_q1gate(stream_, ws_, state_, gp[ii], inv_form, st.p2, n_loc_));
      } else if (kind_is_q2dense(k)) {
        PROF(CAT_UNCOMPUTE, 2, eng_q2gate(stream_, ws_, state_, gp[ii], inv_form, st.p2, st.p1, n_loc_));
      } else {
        PROF(CAT_UNCOMPUTE, 2, eng_q2diag(stream_, ws_, state_, e, true, s2, s1, n_loc_));
      }
      account(1, 1, 2);
      return nullptr;
    }
    if (kind_is_q1(k)) {
      PROF(gdst ? CAT_REV_Q1 : CAT_REV_CONST, 4,
           eng_rev_q1(stream_, ws_, state_, bwd_, gp[ii], inv_form, st.p2, n_loc_, gdst));
    } else if (kind_is_q2dense(k)) {
      PROF(gdst ? CAT_REV_Q2 : CAT_REV_CONST, 4,
           eng_rev_q2(stream_, ws_, state_, bwd_, gp[ii], inv_form, st.p2, st.p1, n_loc_, gdst));
    } else {
      PROF(gdst ? CAT_REV_DIAG : CAT_REV_CONST, 4,
           eng_rev_diag(stream_, ws_, state_, bwd_, e, s2, s1, n_loc_, gdst));
    }
    account(gdst ? 2 : 1, 2, 4);
    return nullptr;
  }

  const char* run_backward(const std::vector<const cplx_t*>& gp, const std::vector<const cplx_t*>& dp,
                           const std::vector<long>& vslot) {
    bool live = false;  // is there an adjoint yet? (bwd_option, src/circuit.rs:276)
    for (size_t si = plan_.steps.size(); si-- > 0;) {
      const qdc::Step& st = plan_.steps[si];
      switch (st.type) {
        case qdc::ST_DENS: {
          size_t sj = si;  // the run of densities at this program point (walking backwards)
          while (sj > 0 && plan_.steps[sj - 1].type == qdc::ST_DENS) sj--;
          QDC_TRY(run_seed_run(sj, si, dp, &live));
          si = sj;
          break;
        }
        case qdc::ST_GATE:
          QDC_TRY(bwd_gate_step(st, gp, vslot, live));
          break;
        case qdc::ST_GATE_K: {
          // no adjoint yet: un-compute only; a variable gate keeps its zero gradient
          const cplx_t* inv = d_kmat_ + gmat_ofs_[st.inst];
          const int k = insts_[st.inst].kind;
          if (!live) QDC_TRY(gate_k_apply(st, state_, inv, CAT_GATE_K_REV));
          else QDC_TRY(gate_k_reverse(st, inv, inv + ((size_t)1 << (2 * st.nk)),
                                      kind_is_var(k) ? d_res_ + kgofs_[st.inst] : nullptr));
          break;
        }
        case qdc::ST_DIAG_K: {
          // forms: the un-compute form, then d, 2^k_loc entries each; no adjoint yet: un-compute only
          const cplx_t* inv = d_kmat_ + gmat_ofs_[st.inst];
          const int k = insts_[st.inst].kind;
          const size_t len = (size_t)1 << qdc::diag_fold_split(st.pk, st.nk, n_loc_, rank_).k_loc;
          if (!live) QDC_TRY(diag_k_apply(st, state_, inv, CAT_DIAG_K_REV));
          else QDC_TRY(diag_k_reverse(st, inv, inv + len, kind_is_var(k) ? d_res_ + kgofs_[st.inst] : nullptr));
          break;
        }
        case qdc::ST_TILE:
#ifndef QDC_F64
          if (tc_step_ok(st)) {
            if (live) QDC_TRY(run_tc_backward(st, gp));
            else QDC_TRY(run_tc_forward(st, gp, true));
            break;
          }
#endif
          if (opt_fuse_ >= 2) {
            // The register-blocked reverse kernel (2 x 16 amplitudes + 32 accumulators per thread)
            // is occupancy-starved and measured slower than the per-gate tile kernel (fuse = 3
            // selects it for experiments); the reverse pass keeps the per-gate tile kernel.
#ifndef QDC_F64
            if (live && opt_fuse_ >= 3) QDC_TRY(run_tile_backward_rb(st, gp, vslot));
            else
#endif
            if (live) QDC_TRY(run_tile_backward(st, gp, vslot, live));
            else QDC_TRY(run_tile_forward_blocked(st, gp, true));
          } else {
            QDC_TRY(run_tile_backward(st, gp, vslot, live));
          }
          break;
        case qdc::ST_SWAP: {
          int gb[3], lp[3];
          const int k = swap_run(si, -1, gb, lp);
          if (k >= 2) {
            PROF(CAT_EXCHANGE, 0, exchange_multi(state_, k, gb, lp));
            if (live) PROF(CAT_EXCHANGE, 0, exchange_multi(bwd_, k, gb, lp));
            si -= (size_t)(k - 1);
          } else {
            PROF(CAT_EXCHANGE, 0, exchange(state_, st.gbit, st.lpos));
            if (live) PROF(CAT_EXCHANGE, 0, exchange(bwd_, st.gbit, st.lpos));
          }
          break;
        }
      }
    }
    return nullptr;
  }

  // ------------------------------------------------------- tiled passes
  // (tile_kernels.cuh)
  const char* run_tile_forward(const qdc::Step& t, const std::vector<const cplx_t*>& gp);
  const char* run_tile_backward(const qdc::Step& t, const std::vector<const cplx_t*>& gp,
                                const std::vector<long>& vslot, bool live);
  const char* run_tile_forward_rb(const qdc::Step& t, const std::vector<const cplx_t*>& gp, bool uncompute);
  const char* run_tile_backward_rb(const qdc::Step& t, const std::vector<const cplx_t*>& gp,
                                   const std::vector<long>& vslot);
  const char* run_tile_forward_rbs(const qdc::Step& t, const std::vector<const cplx_t*>& gp, bool uncompute);
  // Forward / un-compute pass of the default executor (fuse = 2).  Register blocking pays when a block's
  // gates are cheap relative to a shared-memory round trip of the tile (one-qubit and diagonal gates: VQSE-28
  // forward 347 vs 480 ms); for passes dominated by dense two-qubit gates the one-gate-per-sweep pair-lane
  // kernel is faster (28 q brickwork forward 234 vs 264 ms: the blocked kernel's strided block accesses cost
  // it 57 % of its shared wavefronts in bank conflicts, profiles/r1_tile_fwd_rbs_28q_ncu.txt).
  int opt_rb_policy_ = 2;  // 0: never register-block, 1: always, 2: by gate mix (default)
  const char* run_tile_forward_blocked(const qdc::Step& t, const std::vector<const cplx_t*>& gp, bool uncompute) {
    bool blocked = opt_rb_policy_ == 1;
    if (opt_rb_policy_ == 2) {
      int dense_q2 = 0;
      for (int k = 0; k < t.count; k++)
        dense_q2 += kind_is_q2dense(insts_[plan_.tile_steps[t.first + k].inst].kind) ? 1 : 0;
      blocked = 2 * dense_q2 <= t.count;
    }
#ifndef QDC_F64
    if (opt_soa_) {
      if (blocked) return run_tile_forward_rbs(t, gp, uncompute);
      return uncompute ? run_tile_backward(t, gp, std::vector<long>(), false) : run_tile_forward(t, gp);
    }
#endif
    if (blocked) return run_tile_forward_rb(t, gp, uncompute);
    return uncompute ? run_tile_backward(t, gp, std::vector<long>(), false) : run_tile_forward(t, gp);
  }
  void release_tiles();
#ifndef QDC_F64
  // tensor-core fused blocks (tc_exec.cuh)
  void release_tc();
  bool tc_step_ok(const qdc::Step& t) const;
  const char* tc_ensure(size_t image_slots, size_t grad_slots);
  const char* tc_begin(bool backward);
  const char* tc_prepare(const qdc::Step& t, const std::vector<const cplx_t*>& gp, tcb::Params* geo, TcPass* pass);
  const char* tc_launch_block(cplx_t* buf, const tcb::Params& geo, const std::vector<zc>& w, int form, bool launch,
                              tcb::Params* geo_out = nullptr);
  const char* run_tc_forward(const qdc::Step& t, const std::vector<const cplx_t*>& gp, bool uncompute);
  const char* run_tc_backward(const qdc::Step& t, const std::vector<const cplx_t*>& gp);
  const char* tc_finish_backward();
  const std::vector<zc>* tc_gradient(size_t inst) const;
#endif
  // batched densities / seeds (tile_dens_kernels.cuh)
  const char* fill_dens_params(const DensGroup& g, TileDensParams* p, std::vector<int>* tpos);
  const char* run_dens_group(const DensGroup& g, const std::vector<long>& dslot);
  const char* run_seed_group(const DensGroup& g, const std::vector<const cplx_t*>& dp, bool live);
  const char* run_dens_run(size_t first, size_t last, const std::vector<long>& dslot);
  const char* run_seed_run(size_t first, size_t last, const std::vector<const cplx_t*>& dp, bool* live);
  // k-qubit densities / seeds (dens_k_kernels.cuh)
  const char* fill_dens_k_params(const qdc::Step& st, DensKParams* p);
  template <int KQ> const char* launch_dens_k(const DensKParams& p, double* dst);
  template <int KQ> const char* launch_seed_k(const DensKParams& p, const cplx_t* G);
  const char* dens_k(const qdc::Step& st);
  const char* seed_k(const qdc::Step& st, bool live);
  // k-qubit gates (gate_k_kernels.cuh)
  const char* gate_k_forms(const cplx_t* U, int nk, bool nonu, bool reverse, std::vector<cplx_t>* h);
  template <int KQ> const char* launch_gate_k(const DensKParams& p, cplx_t* buf, const cplx_t* At);
  template <int KQ> const char* launch_gate_k_rev(const DensKParams& p, const cplx_t* At, const cplx_t* Bt,
                                                  double* gdst);
  const char* gate_k_apply(const qdc::Step& st, cplx_t* buf, const cplx_t* At, int cat);
  const char* gate_k_reverse(const qdc::Step& st, const cplx_t* At, const cplx_t* Bt, double* gdst);
  // diagonal k-qubit gates (diag_k_kernels.cuh)
  const char* diag_k_forms(const cplx_t* d, const Inst& in, const int* pk, bool reverse, std::vector<cplx_t>* h);
  const char* launch_diag_k(cplx_t* buf, const cplx_t* form, const DiagKPos& p);
  const char* launch_diag_k_rev_whole(const DiagKPos& p, const cplx_t* A, const cplx_t* B, double* gdst);
  template <int NI> const char* launch_diag_k_rev(const DensKParams& dp, const DiagKPos& p, const cplx_t* A,
                                                  const cplx_t* B, double* gdst);
  const char* diag_k_apply(const qdc::Step& st, cplx_t* buf, const cplx_t* form, int cat);
  const char* diag_k_reverse(const qdc::Step& st, const cplx_t* A, const cplx_t* B, double* gdst);
  // physical positions of the plan step of diagonal k-qubit instruction i
  const int* exec_pk(size_t i) const {
    for (const qdc::Step& st : plan_.steps)
      if (st.type == qdc::ST_DIAG_K && st.inst == (int)i) return st.pk;
    return insts_[i].kpos;
  }
  std::vector<char> diag_hilo_;  // diagonal gradient of this instruction came back in (hi,lo) order
  double* tile_partials_ = nullptr;
  size_t tile_partials_cap_ = 0;
};
