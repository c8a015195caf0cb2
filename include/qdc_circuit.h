/* qdc_circuit.h -- circuit-level C ABI of the B200 differentiable statevector
 * engine.  It carries the contract of the reference's `Circuit` pyclass
 * (/root/reference/src/circuit.rs:86-430: builder methods, `run`, `forward`,
 * `backward`) across a plain C boundary, so that a host layer in any language
 * (the reference's Rust/PyO3 `circuit.rs`, or this repo's Python mirror
 * `quantum_differentiable_circuit.Circuit`) can hand a whole program to the
 * GPU instead of one FFI call per instruction (src/circuit.rs:175, 226, 278).
 *
 * All pointers are HOST memory unless stated otherwise.  Gate lists are
 * passed flattened: `gates` holds the matrices back to back in list order,
 * `lens[i]` is the number of complex entries of list element i (4 or 16),
 * `count` the number of list elements.  Results are written (not accumulated)
 * flat, back to back, in the reference's output order.
 *
 * Errors: NULL on success, otherwise a heap message (same convention as
 * qdc_primitives.h).  Messages for the conditions the reference panics on
 * reuse the reference's panic text.
 */
#ifndef QDC_CIRCUIT_H
#define QDC_CIRCUIT_H

#include <stddef.h>
#include <stdint.h>

#include "qdc_primitives.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct qdc_circuit qdc_circuit;

/* Instruction kinds == `enum Instruction`, src/circuit.rs:53-68 (same order),
 * then the densities on 3..6 qubits, which only qdc_circuit_add_dens adds,
 * then the gates on 3..6 qubits, which only qdc_circuit_add_gate adds,
 * then the diagonal gates on 1..6 qubits, which only qdc_circuit_add_gate_diag adds. */
enum qdc_kind {
  QDC_CONST_Q2 = 0, QDC_VAR_Q2 = 1, QDC_CONST_Q2_NONU = 2, QDC_VAR_Q2_NONU = 3,
  QDC_CONST_Q2_DIAG = 4, QDC_VAR_Q2_DIAG = 5,
  QDC_CONST_Q1 = 6, QDC_CONST_Q1_NONU = 7, QDC_VAR_Q1 = 8, QDC_VAR_Q1_NONU = 9,
  QDC_Q2_DENS = 10, QDC_Q1_DENS = 11, QDC_DIFF_Q2_DENS = 12, QDC_DIFF_Q1_DENS = 13,
  QDC_DENS_K = 14, QDC_DIFF_DENS_K = 15,
  QDC_CONST_GATE_K = 16, QDC_VAR_GATE_K = 17, QDC_CONST_GATE_K_NONU = 18, QDC_VAR_GATE_K_NONU = 19,
  QDC_CONST_GATE_K_DIAG = 20, QDC_VAR_GATE_K_DIAG = 21, QDC_CONST_GATE_K_DIAG_NONU = 22, QDC_VAR_GATE_K_DIAG_NONU = 23
};

/* qdc_circuit_count selectors */
enum qdc_count {
  QDC_N_INSTRUCTIONS = 0, QDC_N_CONST_GATES = 1, QDC_N_VAR_GATES = 2,
  QDC_N_DENSITIES = 3,         /* outputs of run()      */
  QDC_N_DIFF_DENSITIES = 4,    /* outputs of forward()  */
  QDC_RUN_OUT_LEN = 5,         /* complex entries written by run()      */
  QDC_FORWARD_OUT_LEN = 6,     /* complex entries written by forward()  */
  QDC_BACKWARD_OUT_LEN = 7     /* complex entries written by backward() */
};

/* Circuit::new, src/circuit.rs:95-103 (state |0..0>; the initial-state copy is
 * materialised lazily, only after set_state_from_host). */
const char* qdc_circuit_new(qdc_circuit** out, size_t qubits_number);
/* Sharded construction (no counterpart in the reference, which is single-GPU):
 * rank r of world = 2^g ranks owns the amplitudes whose top g index bits equal
 * r (the top g PHYSICAL positions are "global").  Gates on local positions and
 * diagonal gates run without communication; a dense gate or a density on a
 * global qubit triggers a qubit-remap swap = one half-shard exchange with the
 * partner rank (NCCL point-to-point over NVLink).  `nccl_unique_id` is the 128
 * byte id from qdc_nccl_unique_id() on rank 0, distributed by the caller.
 * set_state_from_host takes this rank's shard; run/forward/backward return
 * this rank's PARTIAL densities / gradients: the caller sums them over ranks. */
const char* qdc_circuit_new_sharded(qdc_circuit** out, size_t qubits_number, int rank, int world,
                                    const void* nccl_unique_id);
const char* qdc_nccl_unique_id(void* out128);
/* 1 if qubit-remap exchanges run as the fused peer-memory swap kernel (partners'
 * buffers mapped with CUDA IPC over NVLink), 0 if they use NCCL send/recv with
 * pack / unpack passes (option "peer" = 0 forces the latter). */
int qdc_circuit_peer_exchange(const qdc_circuit* c);
const char* qdc_circuit_free(qdc_circuit* c);
/* Circuit::set_state_from_vector, src/circuit.rs:104-106 */
const char* qdc_circuit_set_state_from_host(qdc_circuit* c, const qdc_complex* host_state, size_t len);
/* The 14 builder methods, src/circuit.rs:108-162.  pos1 is ignored for q1 kinds.
 * QDC_DENS_K / QDC_DIFF_DENS_K are refused here (they need qdc_circuit_add_dens), and so are
 * QDC_*_GATE_K (they need qdc_circuit_add_gate) and QDC_*_GATE_K_DIAG* (qdc_circuit_add_gate_diag). */
const char* qdc_circuit_add(qdc_circuit* c, int kind, size_t pos2, size_t pos1);
/* Reduced density matrix on k = 1..6 distinct qubits positions[0..k-1] (positions[0] is the most
 * significant bit of the row and column index), with gradient if `with_grad`:
 *   rho[r, c] = sum_rest psi[r, rest] conj psi[c, rest],   2^k x 2^k, row-major, not normalised.
 * k = 1 and 2 add QDC_(DIFF_)Q1_DENS(positions[0]) and QDC_(DIFF_)Q2_DENS(positions[0], positions[1]);
 * k >= 3 adds QDC_(DIFF_)DENS_K.  Like every density it is a barrier; run / forward return it in program
 * order and backward takes its (conjugated) 4^k-entry cotangent in program order. */
const char* qdc_circuit_add_dens(qdc_circuit* c, const size_t* positions, size_t k, int with_grad);
/* Gate on k = 1..6 distinct qubits positions[0..k-1] (positions[0] is the most significant bit of the
 * row and column index), constant or `variable` (with gradient), unitary or `non_unitary`:
 *   psi'[r, rest] = sum_c U[r, c] psi[c, rest],   U: 2^k x 2^k, row-major, 4^k entries, taken in
 *   program order from the const / var gate lists like every other gate.
 * The reverse pass un-computes with U^dagger (U^-1 for non_unitary, Gauss-Jordan in double precision;
 * a singular pivot fails with "U(i, i) is zero."), returns G[r, c] = sum_rest bwd[r, rest] fwd[c, rest]
 * (4^k entries, no conjugation, like the two-qubit gradient) and pulls the adjoint back with U^T.
 * A variable gate after the last differentiable density has a zero gradient, like every gate kind.
 * k = 1 and 2 add QDC_{CONST,VAR}_Q1[_NONU](positions[0]) and QDC_{CONST,VAR}_Q2[_NONU](positions[0],
 * positions[1]); k >= 3 adds QDC_{CONST,VAR}_GATE_K[_NONU], a barrier like a density: the executor moves
 * no instruction across it. */
const char* qdc_circuit_add_gate(qdc_circuit* c, const size_t* positions, size_t k, int variable,
                                 int non_unitary);
/* Diagonal gate on k = 1..6 distinct qubits positions[0..k-1] (positions[0] is the most significant bit
 * of the index j), constant or `variable` (with gradient), unitary or `non_unitary`:
 *   psi'[j, rest] = d[j] psi[j, rest],   d: 2^k entries, taken in program order from the const / var
 *   gate lists like every other gate.
 * The reverse pass un-computes with conj(d) (1 / d for non_unitary, in double precision; a zero entry
 * fails with "U(j, j) is zero."), returns G[j] = sum_rest bwd[j, rest] fwd[j, rest] (2^k entries, no
 * conjugation, like the two-qubit diagonal's gradient) and pulls the adjoint back with d (U^T = U).
 * A variable gate after the last differentiable density has a zero gradient, like every gate kind.
 * A unitary gate on k = 2 adds QDC_{CONST,VAR}_Q2_DIAG(positions[0], positions[1]); every other case
 * adds QDC_{CONST,VAR}_GATE_K_DIAG[_NONU], a barrier like a density (the executor moves no instruction
 * across it) that needs none of its qubits local on a sharded register: it costs no exchange. */
const char* qdc_circuit_add_gate_diag(qdc_circuit* c, const size_t* positions, size_t k, int variable,
                                      int non_unitary);
size_t qdc_circuit_count(const qdc_circuit* c, int what);

/* Circuit::run, src/circuit.rs:164-212 (all densities, program order). */
const char* qdc_circuit_run(qdc_circuit* c,
                            const qdc_complex* const_gates, const uint32_t* const_lens, size_t n_const,
                            const qdc_complex* var_gates, const uint32_t* var_lens, size_t n_var,
                            qdc_complex* densities_out, size_t out_capacity, size_t* out_len);
/* Circuit::forward, src/circuit.rs:214-264 (Diff* densities only). */
const char* qdc_circuit_forward(qdc_circuit* c,
                                const qdc_complex* const_gates, const uint32_t* const_lens, size_t n_const,
                                const qdc_complex* var_gates, const uint32_t* var_lens, size_t n_var,
                                qdc_complex* densities_out, size_t out_capacity, size_t* out_len);
/* Circuit::backward, src/circuit.rs:266-429.  `dens_grads` are the (already
 * conjugated, src/qdc/circuit.py:193) cotangents of the Diff* densities in
 * program order; the result is one flat gradient per variable gate in program
 * order (4 / 16 / 4 entries). */
const char* qdc_circuit_backward(qdc_circuit* c,
                                 const qdc_complex* dens_grads, const uint32_t* dens_lens, size_t n_dens,
                                 const qdc_complex* const_gates, const uint32_t* const_lens, size_t n_const,
                                 const qdc_complex* var_gates, const uint32_t* var_lens, size_t n_var,
                                 qdc_complex* grads_out, size_t out_capacity, size_t* out_len);

/* QuantizedTensor::get_cpu_state_copy on the circuit's working state,
 * src/quantized_tensor.rs:91-99 (2^n entries). */
const char* qdc_circuit_copy_state_to_host(qdc_circuit* c, qdc_complex* host_state);
/* State I/O (SURVEY.md 8(f) item 4; no reference counterpart beyond
 * get_cpu_state_copy).  One file per rank: a 128-byte header
 *   char magic[8] = "QDCSTAT1"; u32 real_bytes (4|8), n, n_loc, rank, world, reserved;
 *   u8 map[64] (logical qubit -> physical position, 0xFF unused); u8 pad[32]
 * followed by the rank's shard, 2^n_loc raw little-endian interleaved (re, im)
 * pairs in PHYSICAL order (streamed through pinned staging, so a 32 GiB shard
 * needs no 32 GiB host buffer).  save writes the WORKING state (after forward
 * the layout is the plan's final qubit map, recorded in the header); load
 * installs a file in the identity layout as the circuit's INITIAL state, like
 * set_state_from_host.  state_layout reports the current map (n ints). */
const char* qdc_circuit_save_state(qdc_circuit* c, const char* path);
const char* qdc_circuit_load_state(qdc_circuit* c, const char* path);
const char* qdc_circuit_state_layout(const qdc_circuit* c, int* logical_to_physical);
/* DEVICE pointer of the working state (for callers that own device plumbing). */
const char* qdc_circuit_state_device_ptr(qdc_circuit* c, void** device_ptr);
/* Run on a caller-provided cudaStream_t (default: the legacy default stream). */
const char* qdc_circuit_set_stream(qdc_circuit* c, void* cuda_stream);
/* Tunables: "fuse" (0 = one pass per instruction, 1 = tiled multi-gate passes),
 * "profile" (1 = time every launch group with CUDA events), "tile_bits",
 * "low_bits", "max_tile_gates" (geometry of the tiled passes; 0 = default),
 * "peer" (sharded: 1 = peer-memory swap kernel, 0 = NCCL send/recv),
 * "soa" (f32 tile kernels: 1 = pair-lane shared-memory layout, 0 = interleaved). */
const char* qdc_circuit_set_option(qdc_circuit* c, const char* key, long value);
/* Execution statistics of the last run/forward/backward call. */
typedef struct {
  uint64_t kernel_launches;   /* kernels of this library launched */
  uint64_t hbm_passes;        /* full sweeps over a 2^n buffer (read or read+write) */
  uint64_t algorithmic_bytes; /* SURVEY.md section 8(d) accounting */
} qdc_stats;
const char* qdc_circuit_last_stats(const qdc_circuit* c, qdc_stats* out);

/* Per-category device timing of the last call (CUDA events on the executing
 * stream; enable with qdc_circuit_set_option(c, "profile", 1)). */
typedef struct {
  uint64_t launches;          /* timed launch groups in this category */
  double ms;                  /* summed device time */
  uint64_t algorithmic_bytes; /* SURVEY.md 8(d) bytes those launches account for */
} qdc_profile_entry;
int qdc_profile_categories(void);
const char* qdc_profile_category_name(int category);
const char* qdc_circuit_last_profile(const qdc_circuit* c, int category, qdc_profile_entry* out);

/* The pass scheduler as a pure function (no device needed): turns an
 * instruction list into the plan the executor would run for `n` qubits of which
 * `n_loc` are local (n_loc == n: single GPU), with tiled multi-gate passes over
 * `tile_bits` positions (0: none) that always include the `low_bits` lowest.
 * Encoding (int64): per step [type, inst, p2, p1, gbit, lpos, count, nbits]
 * (type 0 gate, 1 density, 2 swap of global bit `gbit` with local position
 * `lpos`, 3 tile pass), a tile pass being followed by count x [inst, p2, p1]
 * and nbits x [position]; terminated by [-1, n, final_map[0..n-1]]. */
const char* qdc_schedule_set_strategy(int tile_strategy); /* tiling of later qdc_schedule calls: 0 first-fit,
                                                           1 window growth, 2 + look-ahead, < 0 library default */
const char* qdc_schedule_set_swap_min_pos(int swap_min_pos); /* lowest position of the remap victims of later qdc_schedule
                                                           calls: >= 0 fixed, -1 library default (4), -2 chosen by the
                                                           scheduler's cost model, as a sharded circuit does */
const char* qdc_schedule(size_t n, size_t n_loc, int tile_bits, int low_bits, int max_tile_gates,
                         const int* kinds, const size_t* pos2, const size_t* pos1, size_t count,
                         int all_densities, int64_t* out, size_t capacity, size_t* out_len);

/* Fused single reverse step on DEVICE buffers (the 4*S kernel):
 * fwd <- U^dagger fwd (or U^-1 fwd when non_unitary), grad (+)= sum bwd (x) fwd,
 * bwd <- U^T bwd.  `gate`/`grad` are HOST pointers; grad is accumulated into
 * like the legacy q*grad symbols, and may be NULL for a constant gate.
 * kind: QDC_VAR_Q1 / QDC_VAR_Q2 / QDC_VAR_Q2_DIAG select the gate shape. */
const char* qdc_reverse_step(qdc_complex* fwd, qdc_complex* bwd, const qdc_complex* gate, qdc_complex* grad,
                             int kind, int non_unitary, size_t pos2, size_t pos1, size_t qubits_number);
/* Fused density seed on DEVICE buffers: bwd (+)= G^T (2 conj fwd)
 * (src/circuit.rs:393-420 in one pass).  K = 2 (q1) or 4 (q2) from kind. */
const char* qdc_density_seed(const qdc_complex* fwd, qdc_complex* bwd, const qdc_complex* dens_grad, int kind,
                             int accumulate, size_t pos2, size_t pos1, size_t qubits_number);

/* Library identification: "f32" or "f64", and the ABI revision. */
const char* qdc_precision(void);
int qdc_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* QDC_CIRCUIT_H */
