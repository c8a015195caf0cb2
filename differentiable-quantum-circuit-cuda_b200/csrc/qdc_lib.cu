// libqdc_b200_{f32,f64}.so -- single translation unit.
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 [-DQDC_F64] -shared ...
// Exports: the 18 legacy symbols (include/qdc_primitives.h) and the circuit
// ABI (include/qdc_circuit.h).  Everything else has hidden visibility.
#include "primitives_abi.cuh"
#include "tile_rb_kernels.cuh"
#include "tile_soa_kernels.cuh"
#include "tile_rb_soa_kernels.cuh"
#include "tile_dens_kernels.cuh"
#include "dens_k_kernels.cuh"
#include "gate_k_kernels.cuh"
#include "diag_k_kernels.cuh"
#include "tc_exec.cuh"

struct qdc_circuit {
  Circuit impl;
  explicit qdc_circuit(int n) : impl(n) {}
};

QDC_EXPORT const char* qdc_precision(void) {
#ifdef QDC_F64
  return "f64";
#else
  return "f32";
#endif
}

QDC_EXPORT int qdc_abi_version(void) { return 5; }

QDC_EXPORT const char* qdc_circuit_new(qdc_circuit** out, size_t qubits_number) {
  if (qubits_number < 1 || qubits_number > 40) return qdc_errf("qubits_number out of range.");
  qdc_circuit* c = new qdc_circuit((int)qubits_number);
  const char* e = c->impl.ensure_state();
  if (e) {
    delete c;
    return e;
  }
  *out = c;
  return nullptr;
}

// Sharded construction: rank r of world = 2^g owns the amplitudes whose top g
// index bits equal r; the NCCL communicator is created from `nccl_unique_id`.
QDC_EXPORT const char* qdc_circuit_new_sharded(qdc_circuit** out, size_t qubits_number, int rank, int world,
                                               const void* nccl_unique_id) {
  if (qubits_number < 1 || qubits_number > 48) return qdc_errf("qubits_number out of range.");
  qdc_circuit* c = new qdc_circuit((int)qubits_number);
  const char* e = c->impl.shard(rank, world, nccl_unique_id);
  if (e) {
    delete c;
    return e;
  }
  *out = c;
  return nullptr;
}

QDC_EXPORT const char* qdc_nccl_unique_id(void* out128) {
  const char* e = qdc::nccl().load();
  if (e) return qdc_errf("%s", e);
  qdc::ncclUniqueId id;
  const int rc = qdc::nccl().GetUniqueId(&id);
  if (rc != 0) return qdc_errf("ncclGetUniqueId failed: %s", qdc::nccl().GetErrorString(rc));
  memcpy(out128, &id, sizeof(id));
  return nullptr;
}

QDC_EXPORT const char* qdc_circuit_free(qdc_circuit* c) {
  delete c;
  return nullptr;
}

QDC_EXPORT const char* qdc_circuit_set_state_from_host(qdc_circuit* c, const cplx_t* host_state, size_t len) {
  return c->impl.set_state_from_host(host_state, len);
}

QDC_EXPORT const char* qdc_circuit_add(qdc_circuit* c, int kind, size_t pos2, size_t pos1) {
  return c->impl.add(kind, pos2, pos1);
}

QDC_EXPORT const char* qdc_circuit_add_dens(qdc_circuit* c, const size_t* positions, size_t k, int with_grad) {
  return c->impl.add_dens(positions, k, with_grad != 0);
}

QDC_EXPORT const char* qdc_circuit_add_gate(qdc_circuit* c, const size_t* positions, size_t k, int variable,
                                            int non_unitary) {
  return c->impl.add_gate(positions, k, variable != 0, non_unitary != 0);
}

QDC_EXPORT const char* qdc_circuit_add_gate_diag(qdc_circuit* c, const size_t* positions, size_t k, int variable,
                                                 int non_unitary) {
  return c->impl.add_gate_diag(positions, k, variable != 0, non_unitary != 0);
}

QDC_EXPORT size_t qdc_circuit_count(const qdc_circuit* c, int what) { return c->impl.count(what); }

QDC_EXPORT const char* qdc_circuit_run(qdc_circuit* c, const cplx_t* cgates, const uint32_t* clens, size_t nc,
                                       const cplx_t* vgates, const uint32_t* vlens, size_t nv, cplx_t* out,
                                       size_t cap, size_t* out_len) {
  return c->impl.sweep(GateList{cgates, clens, nc}, GateList{vgates, vlens, nv}, true, out, cap, out_len);
}

QDC_EXPORT const char* qdc_circuit_forward(qdc_circuit* c, const cplx_t* cgates, const uint32_t* clens,
                                           size_t nc, const cplx_t* vgates, const uint32_t* vlens, size_t nv,
                                           cplx_t* out, size_t cap, size_t* out_len) {
  return c->impl.sweep(GateList{cgates, clens, nc}, GateList{vgates, vlens, nv}, false, out, cap, out_len);
}

QDC_EXPORT const char* qdc_circuit_backward(qdc_circuit* c, const cplx_t* dgrads, const uint32_t* dlens,
                                            size_t nd, const cplx_t* cgates, const uint32_t* clens, size_t nc,
                                            const cplx_t* vgates, const uint32_t* vlens, size_t nv, cplx_t* out,
                                            size_t cap, size_t* out_len) {
  return c->impl.backward(GateList{dgrads, dlens, nd}, GateList{cgates, clens, nc},
                          GateList{vgates, vlens, nv}, out, cap, out_len);
}

// Working state of this rank: 2^(n - log2 world) entries in the CURRENT
// physical layout (identity qubit map before forward and after backward).
QDC_EXPORT const char* qdc_circuit_copy_state_to_host(qdc_circuit* c, cplx_t* host_state) {
  QDC_TRY(c->impl.ensure_state());
  QDC_CUDA(cudaStreamSynchronize(c->impl.stream_));
  QDC_CUDA(cudaMemcpy(host_state, c->impl.state_, c->impl.bytes(), cudaMemcpyDeviceToHost));
  return nullptr;
}

// Checkpoint of this rank's working state / reload as the initial state (circuit.cuh: state I/O).
QDC_EXPORT const char* qdc_circuit_save_state(qdc_circuit* c, const char* path) { return c->impl.save_state(path); }
QDC_EXPORT const char* qdc_circuit_load_state(qdc_circuit* c, const char* path) { return c->impl.load_state(path); }
QDC_EXPORT const char* qdc_circuit_state_layout(const qdc_circuit* c, int* logical_to_physical) {
  c->impl.state_layout(logical_to_physical);
  return nullptr;
}

QDC_EXPORT const char* qdc_circuit_state_device_ptr(qdc_circuit* c, void** device_ptr) {
  QDC_TRY(c->impl.ensure_state());
  *device_ptr = c->impl.state_;
  return nullptr;
}

// 1 when exchanges run as the peer-memory swap kernel (CUDA IPC mapping of the
// partners' buffers succeeded on every rank), 0 when they use NCCL send/recv.
QDC_EXPORT int qdc_circuit_peer_exchange(const qdc_circuit* c) { return c->impl.peer_ok_ && c->impl.opt_peer_; }

QDC_EXPORT const char* qdc_circuit_set_stream(qdc_circuit* c, void* cuda_stream) {
  c->impl.stream_ = (cudaStream_t)cuda_stream;
  return nullptr;
}

QDC_EXPORT const char* qdc_circuit_set_option(qdc_circuit* c, const char* key, long value) {
  if (strcmp(key, "fuse") == 0) c->impl.opt_fuse_ = (int)value;
  else if (strcmp(key, "profile") == 0) c->impl.prof_.on = value != 0;
  else if (strcmp(key, "tile_bits") == 0) c->impl.opt_tile_bits_ = (int)value;
  else if (strcmp(key, "low_bits") == 0) c->impl.opt_low_bits_ = (int)value;
  else if (strcmp(key, "rb_policy") == 0) c->impl.opt_rb_policy_ = (int)value;  // fuse=2 forward: 0 never / 1 always / 2 by gate mix
  else if (strcmp(key, "tile_strategy") == 0) c->impl.opt_tile_strategy_ = (int)value;  // 1 window growth, 0 first-fit
  else if (strcmp(key, "batch_dens") == 0) c->impl.opt_batch_dens_ = (int)value;  // 0: one sweep per density / seed
  else if (strcmp(key, "soa") == 0) c->impl.opt_soa_ = (int)value;    // f32 tile kernels: 0 selects the interleaved-layout kernels
  else if (strcmp(key, "peer") == 0) c->impl.opt_peer_ = (int)value;  // 0: force the NCCL send/recv exchange
  else if (strcmp(key, "multi_swap") == 0) c->impl.opt_multi_swap_ = (int)value;  // 0: one exchange per swapped qubit
  else if (strcmp(key, "auto_swap_pos") == 0) c->impl.opt_auto_swap_pos_ = (int)value;  // 0: remap victims from positions >= 4 only
  else if (strcmp(key, "tc") == 0) {   // f32: tensor-core fused 6-qubit blocks (tc_exec.cuh)
#ifdef QDC_F64
    if (value > 0) return qdc_errf("option \"tc\" exists in the f32 build only.");
#endif
    c->impl.opt_tc_ = (int)value;
  } else if (strcmp(key, "tc_products") == 0) {
    if (value != 6 && value != 8) return qdc_errf("tc_products must be 6 or 8.");
    c->impl.opt_tc_products_ = (int)value;
  } else if (strcmp(key, "tc_rev") == 0) {
    c->impl.opt_tc_rev_ = value != 0;
  } else if (strcmp(key, "max_tile_gates") == 0) {
    if (value < 1 || value > QDC_TILE_MAXG_B) return qdc_errf("max_tile_gates must be in 1..%d.", QDC_TILE_MAXG_B);
    c->impl.opt_max_tile_gates_ = (int)value;
  } else return qdc_errf("Unknown option \"%s\".", key);
  return nullptr;
}

typedef struct {
  uint64_t kernel_launches, hbm_passes, algorithmic_bytes;
} qdc_stats;

QDC_EXPORT const char* qdc_circuit_last_stats(const qdc_circuit* c, qdc_stats* out) {
  out->kernel_launches = c->impl.stats_.kernel_launches;
  out->hbm_passes = c->impl.stats_.hbm_passes;
  out->algorithmic_bytes = c->impl.stats_.algorithmic_bytes;
  return nullptr;
}

typedef struct {
  uint64_t launches;
  double ms;
  uint64_t algorithmic_bytes;
} qdc_profile_entry;

QDC_EXPORT int qdc_profile_categories(void) { return CAT_COUNT; }

QDC_EXPORT const char* qdc_profile_category_name(int cat) {
  return (cat >= 0 && cat < CAT_COUNT) ? kProfCatNames[cat] : "";
}

QDC_EXPORT const char* qdc_circuit_last_profile(const qdc_circuit* c, int cat, qdc_profile_entry* out) {
  if (cat < 0 || cat >= CAT_COUNT) return qdc_errf("Unknown profile category %d.", cat);
  out->launches = c->impl.prof_.cats[cat].launches;
  out->ms = c->impl.prof_.cats[cat].ms;
  out->algorithmic_bytes = c->impl.prof_.cats[cat].alg_bytes;
  return nullptr;
}

// ---- scheduler as a pure function (no device needed) ---------------------
// Encoding of the plan, all int64, one record per step:
//   [type, inst, p2, p1, gbit, lpos, count, nbits] then, for TILE steps,
//   count x [inst, p2, p1] followed by nbits x [physical bit].
// After the last step: [-1, n, final_map[0..n-1]].
static int g_schedule_tile_strategy = -1;  // < 0: the library default

// Tiling strategy used by the following qdc_schedule() calls (0 first-fit, 1 window growth, 2 + look-ahead;
// < 0 restores the default).  Lets the CPU suite check every strategy without a device.
QDC_EXPORT const char* qdc_schedule_set_strategy(int tile_strategy) {
  g_schedule_tile_strategy = tile_strategy;
  return nullptr;
}

// Lowest position of the remap victims for the following qdc_schedule() calls: >= 0 fixed, -1 the library default (4),
// -2 chosen by the cost model of scheduler.hpp (what a sharded Circuit does; tile_bits == 6 selects the tensor-core
// pass time).  Lets the CPU suite check those plans without a device.
static int g_schedule_swap_min_pos = -1;
QDC_EXPORT const char* qdc_schedule_set_swap_min_pos(int swap_min_pos) {
  if (swap_min_pos < -2) return qdc_errf("swap_min_pos must be >= -2.");
  g_schedule_swap_min_pos = swap_min_pos;
  return nullptr;
}

QDC_EXPORT const char* qdc_schedule(size_t n, size_t n_loc, int tile_bits, int low_bits, int max_tile_gates,
                                    const int* kinds, const size_t* pos2, const size_t* pos1, size_t count,
                                    int all_densities, int64_t* out, size_t cap, size_t* out_len) {
  std::vector<qdc::SchedInst> si(count);
  for (size_t i = 0; i < count; i++) {
    const int k = kinds[i];
    if (k < 0 || k > K_DIFF_Q1_DENS) return qdc_errf("Unknown instruction kind %d.", k);
    si[i].kind_class = Circuit::sched_class(k);
    si[i].q2 = (int)pos2[i];
    si[i].q1 = (kind_is_q1(k) || kind_is_q1_dens(k)) ? -1 : (int)pos1[i];
    si[i].skip = kind_is_dens(k) && !all_densities && !kind_is_diff_dens(k);
  }
  qdc::SchedOptions so;
  so.n = (int)n;
  so.n_loc = (int)n_loc;
  so.tile_bits = tile_bits;
  so.low_bits = low_bits;
  if (max_tile_gates > 0) so.max_tile_gates = max_tile_gates;
  if (g_schedule_tile_strategy >= 0) so.tile_strategy = g_schedule_tile_strategy;
  if (g_schedule_swap_min_pos >= 0) so.swap_min_pos = g_schedule_swap_min_pos;
  qdc::Plan plan;
  if (g_schedule_swap_min_pos == -2) {
    qdc::CostModel cm;
    cm.amp_bytes = (int)sizeof(cplx_t);
    cm.vec_log2 = QDC_LV;
    if (tile_bits == 6) cm.tile_ms = 59;
    plan = qdc::schedule_best(si, so, cm, nullptr);
  } else {
    qdc::Scheduler sch(si, so);
    plan = sch.run();
  }
  if (!plan.ok) return qdc_errf("the program cannot be scheduled on %zu local qubits per rank.", n_loc);
  std::vector<int64_t> enc;
  for (const qdc::Step& st : plan.steps) {
    const int64_t rec[8] = {st.type, st.inst, st.p2, st.p1, st.gbit, st.lpos, st.count, st.tb_count};
    enc.insert(enc.end(), rec, rec + 8);
    if (st.type == qdc::ST_TILE) {
      for (int k = 0; k < st.count; k++) {
        const qdc::Step& g = plan.tile_steps[st.first + k];
        enc.push_back(g.inst);
        enc.push_back(g.p2);
        enc.push_back(g.p1);
      }
      for (int k = 0; k < st.tb_count; k++) enc.push_back(plan.tile_bits[st.tb_first + k]);
    }
  }
  enc.push_back(-1);
  enc.push_back((int64_t)n);
  for (int q = 0; q < (int)n; q++) enc.push_back(plan.final_map[q]);
  *out_len = enc.size();
  if (enc.size() > cap) return qdc_errf("plan buffer too small: %zu < %zu.", cap, enc.size());
  memcpy(out, enc.data(), enc.size() * sizeof(int64_t));
  return nullptr;
}

QDC_EXPORT const char* qdc_reverse_step(cplx_t* fwd, cplx_t* bwd, const cplx_t* gate, cplx_t* grad, int kind,
                                        int non_unitary, size_t pos2, size_t pos1, size_t n) {
  const int inv_form = non_unitary ? FORM_INV : FORM_CONJ_TR;
  double* dst = nullptr;
  if (grad) {
    QDC_TRY(ws_ensure(g_legacy_ws, 1));
    dst = g_legacy_ws.red_out;
  }
  if (kind_is_q1(kind)) {
    QDC_TRY(eng_rev_q1(0, g_legacy_ws, fwd, bwd, gate, inv_form, (int)pos2, (int)n, dst));
    return grad ? fetch_and_accumulate(8, false, false, grad) : nullptr;
  }
  if (kind_is_q2dense(kind)) {
    QDC_TRY(eng_rev_q2(0, g_legacy_ws, fwd, bwd, gate, inv_form, (int)pos2, (int)pos1, (int)n, dst));
    return grad ? fetch_and_accumulate(32, true, pos2 < pos1, grad) : nullptr;
  }
  if (kind_is_diag(kind)) {
    QDC_TRY(eng_rev_diag(0, g_legacy_ws, fwd, bwd, gate, (int)pos2, (int)pos1, (int)n, dst));
    return grad ? fetch_and_accumulate(8, false, false, grad) : nullptr;
  }
  return qdc_errf("qdc_reverse_step: kind %d is not a gate.", kind);
}

QDC_EXPORT const char* qdc_density_seed(const cplx_t* fwd, cplx_t* bwd, const cplx_t* dens_grad, int kind,
                                        int accumulate, size_t pos2, size_t pos1, size_t n) {
  if (kind_is_q1(kind) || kind_is_q1_dens(kind))
    return eng_seed_q1(0, g_legacy_ws, fwd, bwd, dens_grad, (int)pos2, (int)n, accumulate != 0);
  return eng_seed_q2(0, g_legacy_ws, fwd, bwd, dens_grad, (int)pos2, (int)pos1, (int)n, accumulate != 0);
}
