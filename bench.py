#!/usr/bin/env python
"""Headline benchmark: fwd+bwd gate-applies/sec of a random brickwork circuit.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--qubits 32] [--depth 100] [--precision f32] [--fuse 1]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[3], SURVEY.md 8(d) item 4): n-qubit brickwork of
depth D -- layer l applies `add_q2_var_gate(i+1, i)` for i = l mod 2, l mod 2 + 2, ...
-- Haar-random 4x4 gates (NumPy default_rng(1234)), initial state |0..0>, loss
drivers `get_q2_dens_op_with_grad(i+1, i)` on every even i with a fixed random
Hermitian cotangent.  One STEP = one `Circuit.forward` + one `Circuit.backward`
through the reference-facing API (host NumPy gate lists in, host densities and
per-gate gradients out), i.e. the call a user of the reference makes.

Metric: gate-applies/s = (#gate instructions) / (time of forward + backward).
  value : timed on the device with CUDA events around the K steps.
  e2e   : wall clock around the same public-API calls (host marshalling, H2D of
          the gate matrices as kernel parameters, D2H of densities/gradients).
The state is generated on the device by the API itself (|0..0>, as in the
reference's Circuit::new); the host inputs of the path are the gate lists.

`--impl reference` drives the reference's own CUDA library (oracle/_ref, built
unmodified from /root/reference/src/primitives.cu) with the exact call sequence
of its Rust `Circuit` (oracle/ref_replay.py) on a depth-bounded sample of the
same workload; the reference has no CPU implementation of the path.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "fwd+bwd gate-applies/sec"
UNIT = "gate-applies/s"


# ------------------------------------------------------------------ workload
def haar(rng, k):
    z = rng.normal(size=(k, k)) + 1j * rng.normal(size=(k, k))
    q, r = np.linalg.qr(z)
    return (q * (np.diag(r) / np.abs(np.diag(r)))).reshape(-1)


def brickwork_program(n, depth):
    """[(pos2, pos1)] of the gate instructions and of the trailing densities."""
    gates = []
    for layer in range(depth):
        for i in range(layer % 2, n - 1, 2):
            gates.append((i + 1, i))
    dens = [(i + 1, i) for i in range(0, n - 1, 2)]
    return gates, dens


def build_brickwork(circuit, n, depth):
    gates, dens = brickwork_program(n, depth)
    for p2, p1 in gates:
        circuit.add_q2_var_gate(p2, p1)
    for p2, p1 in dens:
        circuit.get_q2_dens_op_with_grad(p2, p1)
    return len(gates), len(dens)


def brickwork_inputs(n, depth, dtype):
    rng = np.random.default_rng(1234)
    gates, dens = brickwork_program(n, depth)
    var = [haar(rng, 4).astype(dtype) for _ in gates]
    cts = []
    for _ in dens:
        a = rng.normal(size=(4, 4)) + 1j * rng.normal(size=(4, 4))
        cts.append(((a + a.conj().T) / 2).astype(dtype))
    return var, cts


def vqse_program(n, layers):
    """example_vqse_ising.py:66-79: per layer n ring ZZ diagonal gates + n X rotations; n ring densities."""
    prog = []
    for _ in range(layers):
        for i in range(n - 1):
            prog.append(("diag", i, i + 1))
        prog.append(("diag", 0, n - 1))
        for i in range(n):
            prog.append(("q1", i, -1))
    dens = [(i, i + 1) for i in range(n - 1)] + [(0, n - 1)]
    return prog, dens


def build_vqse(circuit, n, layers):
    prog, dens = vqse_program(n, layers)
    for kind, a, b in prog:
        if kind == "diag":
            circuit.add_q2_var_gate_diag(a, b)
        else:
            circuit.add_q1_var_gate(a)
    for a, b in dens:
        circuit.get_q2_dens_op_with_grad(a, b)
    return len(prog), len(dens)


def vqse_inputs(n, layers, dtype):
    """Gates of example_vqse_ising.py:15-28 from 2*layers N(0,1) parameters (seed 42); cotangent = h^T of the
    transverse-field Ising two-site term (:86-93)."""
    rng = np.random.default_rng(42)
    params = rng.normal(size=2 * layers)
    var = []
    for l in range(layers):
        g, b = params[2 * l], params[2 * l + 1]
        zz = np.array([np.exp(-1j * g), np.exp(1j * g), np.exp(1j * g), np.exp(-1j * g)], dtype=dtype)
        x = np.array([np.cos(b), -1j * np.sin(b), -1j * np.sin(b), np.cos(b)], dtype=dtype)
        var += n * [zz] + n * [x]
    sz = np.diag([1.0, -1.0]); sx = np.array([[0, 1.0], [1.0, 0]]); eye = np.eye(2)
    k = lambda a, b: np.tensordot(a, b, axes=0).transpose(0, 2, 1, 3).reshape(4, 4)  # noqa: E731
    h = (-k(sz, sz) - 0.5 * (k(sx, eye) + k(eye, sx))).astype(dtype)
    _, dens = vqse_program(n, layers)
    return var, [h.T.copy() for _ in dens]


# -------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"),
                                   r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------ CPU baseline
def _cpu_baseline_numpy(budget_s):
    """The oracle (NumPy port of the path) on one core: fwd+bwd of brickwork gates at 22 qubits."""
    from oracle import statevector as sv
    n = 22
    rng = np.random.default_rng(1234)
    dtype = np.complex64
    psi = sv.standard_state(n, dtype)
    gates, _ = brickwork_program(n, 8)    # the forward loop stops at budget / 3
    mats = [haar(rng, 4).astype(dtype) for _ in gates]
    t0 = time.perf_counter()
    done = 0
    for (p2, p1), g in zip(gates, mats):   # forward
        psi = sv.q2gate_fast(psi, g, p2, p1)
        done += 1
        if time.perf_counter() - t0 > budget_s / 3:
            break
    bwd = sv.conj_and_double(psi)
    for (p2, p1), g in list(zip(gates, mats))[:done][::-1]:   # backward: un-compute, grad, adjoint
        psi = sv.q2gate_fast(psi, sv.q2_conj_tr(g), p2, p1)
        sv.q2grad(psi, bwd, p2, p1)
        bwd = sv.q2gate_fast(bwd, sv.q2_tr(g), p2, p1)
    dt = time.perf_counter() - t0
    return n, done, dt


def _torch_apply_adjacent(x, g, lo, n):
    """q2 gate (4x4 torch tensor, reference index convention) on the adjacent pair (lo + 1, lo) of a torch state."""
    import torch
    return torch.matmul(g, x.view(1 << (n - lo - 2), 4, 1 << lo)).reshape(-1)


def _cpu_baseline_torch(budget_s):
    """The same algorithm (apply / un-compute with U^dagger / gradient outer product / pull back with U^T) as
    batched 4x4 matmuls on torch CPU tensors with all host threads: fwd+bwd of brickwork gates at 24 qubits."""
    import torch
    n = 24
    rng = np.random.default_rng(1234)
    gates, _ = brickwork_program(n, 40)   # more than the time budget admits: the forward loop stops at budget / 4
    mats = [torch.tensor(haar(rng, 4).reshape(4, 4), dtype=torch.complex64) for _ in gates]
    psi = torch.zeros(1 << n, dtype=torch.complex64)
    psi[0] = 1

    def apply(x, g, lo):
        return _torch_apply_adjacent(x, g, lo, n)

    t0 = time.perf_counter()
    done = 0
    for (p2, p1), g in zip(gates, mats):
        psi = apply(psi, g, p1)
        done += 1
        if time.perf_counter() - t0 > budget_s / 4:
            break
    bwd = 2 * psi.conj()
    for (p2, p1), g in list(zip(gates, mats))[:done][::-1]:
        psi = apply(psi, g.conj().T.contiguous(), p1)
        torch.einsum("apc,aqc->pq", bwd.view(1 << (n - p1 - 2), 4, 1 << p1), psi.view(1 << (n - p1 - 2), 4, 1 << p1))
        bwd = apply(bwd, g.T.contiguous(), p1)
    dt = time.perf_counter() - t0
    return n, done, dt, torch.get_num_threads()


def cpu_baseline(n_target, budget_s=12.0):
    """CPU restatements of the path timed on the host (the reference has no CPU implementation): the NumPy oracle
    on one core and a torch port on all host threads, each on a reduced register (the 2^32-amplitude state does not
    fit a bounded CPU run), scaled to the target size by the amplitude ratio.  The faster one is reported."""
    n1, done1, dt1 = _cpu_baseline_numpy(budget_s)
    r1 = done1 / dt1 * 2.0 ** (n1 - n_target)
    note1 = (f"oracle (NumPy, 1 core) fwd+bwd of {done1} brickwork gates at {n1} qubits complex64 in {dt1:.1f}s "
             f"= {done1 / dt1:.3g} gate-applies/s")
    try:
        n2, done2, dt2, threads = _cpu_baseline_torch(budget_s)
        r2 = done2 / dt2 * 2.0 ** (n2 - n_target)
        note2 = (f"torch-CPU port ({threads} threads of {os.cpu_count()} cores) fwd+bwd of {done2} brickwork gates at "
                 f"{n2} qubits complex64 in {dt2:.1f}s = {done2 / dt2:.3g} gate-applies/s")
    except Exception as e:  # noqa: BLE001
        r2, threads, note2 = 0.0, 1, f"torch-CPU port failed: {e}"
    best, cores = (r2, threads) if r2 > r1 else (r1, 1)
    return {"value": best, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{note2}; {note1}; both scaled by the amplitude ratio to {n_target} qubits, the faster reported"}


# ------------------------------------------------------------------- arms
def dist_setup(n_gpus):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


# FP32/FP64-pipe work of one gate per amplitude, forward (complex multiply-accumulates x 4 real FMA); the reverse
# step of a gate (un-compute, gradient outer product, adjoint pull-back) costs three times that.
FMA_PER_AMP_FWD = {"q2": 16, "q1": 8, "diag": 4}


def workload_kinds(workload, n, depth):
    if workload == "vqse":
        return [("diag" if k == "diag" else "q1") for k, _, _ in vqse_program(n, depth)[0]]
    return ["q2"] * len(brickwork_program(n, depth)[0])


def make_circuit(args, world, n_total, precision, workload, depth, opts=None):
    """Circuit of the public API + its host inputs for one workload."""
    pkg = importlib.import_module("differentiable-quantum-circuit-cuda_b200")
    dtype = np.complex64 if precision == "f32" else np.complex128
    if world > 1:
        sharded = importlib.import_module("differentiable-quantum-circuit-cuda_b200.sharded")
        circ = sharded.ShardedCircuit(n_total, precision=precision)
    elif args.fusion:
        circ = pkg.FusedCircuit(n_total, precision=precision)
    else:
        circ = pkg.Circuit(n_total, precision=precision)
    o = {"fuse": args.fuse, "profile": 1}
    for key, val in (("tile_bits", args.tile_bits), ("low_bits", args.low_bits), ("max_tile_gates", args.max_tile_gates)):
        if val:
            o[key] = val
    if world > 1:
        o["peer"] = args.peer
    if precision == "f32":
        o["soa"] = args.soa
    if precision == "f32" and args.tc >= 0:
        o["tc"] = args.tc
    if precision == "f32" and args.tc_rev >= 0:
        o["tc_rev"] = args.tc_rev
    if precision == "f32" and args.tc_products > 0:
        o["tc_products"] = args.tc_products
    for key, val in (("rb_policy", args.rb_policy), ("batch_dens", args.batch_dens),
                     ("tile_strategy", args.tile_strategy)):
        if val >= 0:
            o[key] = val
    o.update(opts or {})
    for key, val in o.items():
        circ.set_option(key, val)
    if workload == "vqse":
        n_gates, n_dens = build_vqse(circ, n_total, depth)
        var, cts = vqse_inputs(n_total, depth, dtype)
        if world == 1:
            circ.set_state_from_vector((np.ones(1 << n_total) / np.sqrt(float(1 << n_total))).astype(dtype))
    else:
        n_gates, n_dens = build_brickwork(circ, n_total, depth)
        var, cts = brickwork_inputs(n_total, depth, dtype)
    return circ, n_gates, n_dens, var, [c.conj() for c in cts]


def parity_check(args, world, rank, precision, workload, n_small, depth_small):
    """Before timing: the executor exactly as benchmarked (same options, same world size) on a small register
    against the per-gate streaming executor (fuse = 0) on ONE GPU -- rank 0's own single-GPU run when sharded.
    Largest deviation of any density / gradient entry, relative to the largest entry."""
    g = world.bit_length() - 1
    n = n_small + g
    circ, _, _, var, cts = make_circuit(args, world, n, precision, workload, depth_small)
    dens = circ.forward([], var)
    grads = circ.backward(cts, [], var)
    del circ
    out = None
    if rank == 0:
        ref, _, _, var, cts = make_circuit(args, 1, n, precision, workload, depth_small, {"fuse": 0})
        dens_r = ref.forward([], var)
        grads_r = ref.backward(cts, [], var)
        del ref
        dscale = max(float(np.abs(x).max()) for x in dens_r)
        gscale = max(float(np.abs(x).max()) for x in grads_r)
        out = {"against": "per-gate streaming executor (fuse=0) on one GPU, same circuit family",
               "qubits": n, "depth": depth_small, "world": world,
               "max_rel_err_density": max(float(np.abs(a - b).max()) for a, b in zip(dens, dens_r)) / dscale,
               "max_rel_err_gradient": max(float(np.abs(a - b).max()) for a, b in zip(grads, grads_r)) / gscale,
               "tolerance": 1e-5 if precision == "f32" else 1e-12}
        out["ok"] = bool(max(out["max_rel_err_density"], out["max_rel_err_gradient"]) < out["tolerance"])
    return out


def timed_steps(circ, var, cts_conj, warmup, steps, barrier, sampler=None):
    import torch
    for _ in range(warmup):
        circ.forward([], var)
        circ.backward(cts_conj, [], var)
    if sampler is not None:
        sampler.start()
    launches, prof = 0, {}
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    for _ in range(steps):
        dens = circ.forward([], var)
        s_f, p_f = circ.last_stats(), circ.last_profile()
        grads = circ.backward(cts_conj, [], var)
        s_b, p_b = circ.last_stats(), circ.last_profile()
        launches += s_f["kernel_launches"] + s_b["kernel_launches"]
        for p in (p_f, p_b):
            for k, v in p.items():
                e = prof.setdefault(k, {"launches": 0, "ms": 0.0, "algorithmic_bytes": 0})
                for kk in e:
                    e[kk] += v[kk]
    ev1.record()
    barrier()
    wall = time.perf_counter() - t0
    return ev0.elapsed_time(ev1), wall, prof, launches, dens, grads


def load_peaks():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        peaks = {}
    peak = float(peaks.get("hbm_gbs", 6650.0))
    src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    return peak, src, float(peaks.get("sm_max_mhz", 1965.0))


def roofline_block(prof, dev_ms, steps, precision, local_qubits, kinds, clocks, tc_rev=True, tc_products=6):
    """Dominant kernel = the category with the most device time.  `achieved` / `frac` follow SURVEY 8(d):
    algorithmic bytes (2*S forward, 4*S reverse PER GATE) over the launch time against the measured HBM copy
    peak -- above 1 when a launch applies several gates.  The binding resource of the tiled passes is the
    FP32 (FP64) FMA pipe, reported beside it with the real DRAM rate."""
    if not prof:
        return None
    peak, peak_src, sm_max_mhz = load_peaks()
    name, e = max(prof.items(), key=lambda kv: kv[1]["ms"])
    sec = e["ms"] * 1e-3
    achieved = e["algorithmic_bytes"] / sec / 1e9
    itemsize = 8 if precision == "f32" else 16
    S = itemsize << local_qubits
    r = {"bound": "hbm", "kernel": name, "achieved": round(achieved, 1), "peak": peak, "peak_source": peak_src,
         "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": None, "launches": e["launches"],
         "avg_launch_ms": round(e["ms"] / e["launches"], 4),
         "algorithmic_bytes_per_launch": e["algorithmic_bytes"] // e["launches"],
         "share_of_step": round(e["ms"] / dev_ms, 4)}
    if name in ("tile_bwd", "tile_fwd"):
        mult = 3 if name == "tile_bwd" else 1
        fma = mult * sum(FMA_PER_AMP_FWD[k] for k in kinds) * float(1 << local_qubits) * steps
        lanes = 128 if precision == "f32" else 64     # FMA per clock per SM
        clk = sm_max_mhz
        if clocks and clocks.get("sm_mhz"):
            clk = min(clk, float(clocks["sm_mhz"]))
        pipe_peak = 148 * lanes * sm_max_mhz * 1e6 / 1e12
        r["bound"] = "fp32" if precision == "f32" else "fp64"
        r["fp_tfma_s"] = round(fma / sec / 1e12, 2)
        r["fp_peak_tfma_s"] = round(pipe_peak, 2)
        r["fp32_frac" if precision == "f32" else "fp64_frac"] = round(fma / sec / 1e12 / pipe_peak, 4)
        r["fp_peak_note"] = (f"148 SMs x {lanes} FMA/clk x {sm_max_mhz:.0f} MHz (clocks.max.sm); median SM clock under "
                             f"load {clk:.0f} MHz")
        passes = 4 if name == "tile_bwd" else 2      # a launch reads + writes the state (and the adjoint) once
        r["traffic"] = passes * S
        r["traffic_source"] = ("= %d*S per launch whatever the number of fused gates; ncu dram__bytes_read+write of "
                               "one launch: profiles/r2_traffic.json (r1: 137.4 GB = 4*S at 32 q)" % passes)
        r["dram_gbs"] = round(passes * S * e["launches"] / sec / 1e9, 1)
        r["dram_frac"] = round(r["dram_gbs"] / peak, 4)
        r["gates_per_launch"] = round(r["algorithmic_bytes_per_launch"] / float(passes * S), 2)
    if name in ("tc_bwd", "tc_fwd"):
        # tensor-core fused blocks (csrc/tc_block.cuh, tc_rev.cuh): one 64 x 64 block per HBM sweep.  Reverse step of a
        # block = ONE fused sweep over state and adjoint (4*S of real traffic); with option tc_rev = 0 un-compute (2*S) +
        # block gradient (2*S read) + adjoint pull-back (2*S) = 6*S.
        passes = (4 if tc_rev else 6) if name == "tc_bwd" else 2
        alg = 4 if name == "tc_bwd" else 2
        tiles = float(1 << (local_qubits - 12))
        mma_flop = 2.0 * 128 * 64 * 16                     # one tcgen05.mma of the block kernel (M 128, N 64, K 16)
        blk = 8 * tc_products                              # MMAs of one block product (6 or 8 slice products x K / 16)
        per_tile = (2 * blk + 24 * 2) * mma_flop if name == "tc_bwd" else blk * mma_flop
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:  # noqa: BLE001
            pass
        tpeak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
        r["bound"] = "hbm"
        r["traffic"] = passes * S
        r["traffic_source"] = ("= %d*S per block (state%s read + written once per kernel of the block)"
                               % (passes, " and adjoint" if name == "tc_bwd" else ""))
        r["dram_gbs"] = round(passes * S * e["launches"] / sec / 1e9, 1)
        r["dram_frac"] = round(r["dram_gbs"] / peak, 4)
        r["tensor_tflops"] = round(per_tile * tiles * e["launches"] / sec / 1e12, 1)
        r["tensor_peak_tflops"] = tpeak
        r["tensor_frac"] = round(r["tensor_tflops"] / tpeak, 4)
        r["tensor_note"] = ("bf16 tcgen05.mma on exact 9-bit slices of the f32 data: %d instructions of 128 x 64 x 16 per block "
                            "product and 2^12-amplitude tile%s; peak = measured cuBLAS bf16 (sustained)"
                            % (blk, " (two block products + 24 of 128 x 128 x 16 for the block gradient)" if name == "tc_bwd" else ""))
        r["gates_per_launch"] = round(r["algorithmic_bytes_per_launch"] / float(alg * S), 2)
        r["binding_resource"] = ("neither roof alone: real DRAM traffic runs at dram_frac of the measured copy peak and the tcgen05 MMAs at "
                                 "tensor_frac of the measured cuBLAS bf16 rate; ncu (profiles/r2_tc_rev_28q_v7_ncu.txt) shows the L1 data pipe, "
                                 "shared by the tensor-core operand reads and the fill / drain traffic, at 64 % and the board under its "
                                 "power cap (see clocks); frac > 1 is the ~9 gates fused per sweep")
    return r


def dump_outputs(out_dir, dens, grads):
    """What a caller of the timed path receives from its last step, as real arrays with a trailing (real, imag) axis:
    densities.npy (densities x 4 x 4 x 2) and gradients.npy (gates x gate entries x 2), float32 for f32 and float64
    for f64.  The inputs are seeded, so two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, z in (("densities", np.stack([np.asarray(d) for d in dens])),
                    ("gradients", np.stack([np.asarray(g).reshape(-1) for g in grads]))):
        np.save(os.path.join(out_dir, name + ".npy"), np.stack([z.real, z.imag], axis=-1))


def run_workload(args, world, rank, local, precision, workload, local_qubits, depth, warmup, steps, barrier,
                 sample_clocks, check_sizes, dump_dir=None):
    """Parity check, then the timed steps of one workload; returns the JSON fields (rank 0) or None.  With dump_dir,
    rank 0 also writes the outputs of the last timed step there (dump_outputs)."""
    import torch
    g = world.bit_length() - 1
    n_total = local_qubits + g
    check = parity_check(args, world, rank, precision, workload, *check_sizes) if not args.no_check else None
    barrier()
    circ, n_gates, n_dens, var, cts_conj = make_circuit(args, world, n_total, precision, workload, depth)
    dtype = np.complex64 if precision == "f32" else np.complex128
    sampler = ClockSampler(local) if (sample_clocks and rank == 0) else None
    dev_ms, wall, prof, launches, dens, grads = timed_steps(circ, var, cts_conj, warmup, steps, barrier, sampler)
    clocks = sampler.stop() if sampler is not None else None
    peer = circ.peer_exchange if world > 1 else None
    del circ
    torch.cuda.empty_cache()
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([dev_ms, wall], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall = float(t[0]), float(t[1])
    if rank != 0:
        return None
    peak, _, _ = load_peaks()
    kinds = workload_kinds(workload, n_total, depth)
    total_alg = sum(e["algorithmic_bytes"] for e in prof.values())
    h2d = sum(v.nbytes for v in var) * 2 + sum(c.nbytes for c in cts_conj)   # gates go in twice (fwd, bwd)
    d2h = n_dens * 16 * var[0].itemsize + sum(v.nbytes for v in var)
    # Work unit = one gate applied to one 2^local_qubits-amplitude shard.  A sharded run applies every
    # gate to `world` shards, so the whole-job aggregate is world * gates / time (weak scaling: per-GPU
    # work per gate is fixed; ideal aggregate grows linearly with the number of GPUs).
    value = world * n_gates * steps / (dev_ms * 1e-3)
    check = dict(check or {})
    check.update({"trace_density0": float(np.trace(dens[0]).real),
                  "grad_norm": float(np.sqrt(sum(np.vdot(x, x).real for x in grads)))})
    if dump_dir:
        dump_outputs(dump_dir, dens, grads)
    return {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": round(dev_ms / steps, 3), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": precision, "data": "synthetic",
        "full_state_gate_applies_per_s": round(n_gates * steps / (dev_ms * 1e-3), 3),
        "config": {"workload": f"{workload}-{n_total}q-depth{depth}-{precision}", "qubits": n_total,
                   "local_qubits": local_qubits, "depth": depth, "gates": n_gates, "densities": n_dens,
                   "state_bytes_per_gpu": int(np.dtype(dtype).itemsize) << local_qubits,
                   "unit_note": "one gate-apply = one gate applied (fwd+bwd) to one 2^local_qubits-amplitude shard; "
                                "an N-GPU run applies each gate to N shards; full_state_gate_applies_per_s counts each "
                                "gate once whatever N (the figure to set against a one-GPU reference run)",
                   "l2": "inputs (state + adjoint) far larger than L2; no flush needed" if local_qubits >= 26 else
                         "state + adjoint fit L2 at this size",
                   "exchange": (("peer-memory swap kernel (NVLink, CUDA IPC)" if peer else
                                 "NCCL send/recv + pack/unpack") if world > 1 else None),
                   "gate_fusion": bool(args.fusion and world == 1),
                   "executor": ["one pass per gate", "tiled multi-gate passes",
                                "tiled multi-gate passes, forward kernel (register-blocked or per gate) by gate mix"][args.fuse]
                               + (", pair-lane smem layout" if precision == "f32" and args.soa and args.fuse else "")
                               + (", tensor-core fused 6-qubit blocks (tcgen05, exact bf16 slices)"
                                  if "tc_fwd" in prof or "tc_bwd" in prof else "")},
        "effective_hbm_gbs": round(total_alg * world / (dev_ms * 1e-3) / 1e9, 1),
        "effective_hbm_frac": round(total_alg / (dev_ms * 1e-3) / 1e9 / peak, 4),
        "roofline": roofline_block(prof, dev_ms, steps, precision, local_qubits, kinds, clocks, tc_rev=args.tc_rev != 0,
                                   tc_products=args.tc_products or 6),
        "profile_ms": {k: round(v["ms"], 2) for k, v in sorted(prof.items())},
        "e2e": {"value": round(world * n_gates * steps / wall, 3), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h)},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "check": check,
    }


def run_ours(args):
    import torch
    rank, world, local = dist_setup(args.gpus)

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    small = (24, 8) if args.workload == "brickwork" else (22, 3)
    out = run_workload(args, world, rank, local, args.precision, args.workload, args.qubits, args.depth, args.warmup,
                       args.steps, barrier, True, small, args.dump_outputs)
    # the other single-GPU BASELINE.json configs, each with its own roofline and parity check
    if world == 1 and args.secondary and args.workload == "brickwork" and args.precision == "f32" and args.qubits == 32:
        sec = {}
        try:
            r = run_workload(args, 1, 0, local, "f32", "vqse", 28, 26, 3, 5, barrier, False, (22, 3))
            sec["vqse-28q-26layers-f32"] = r
            r = run_workload(args, 1, 0, local, "f64", "brickwork", 32, 100, 1, 1, barrier, False, (24, 8))
            r["config"]["note"] = "1 warm-up + 1 timed step (52 s each): bounded so the default run stays within minutes"
            sec["brickwork-32q-depth100-f64"] = r
        except Exception as e:  # noqa: BLE001
            sec["error"] = repr(e)
        if rank == 0:
            out["secondary"] = sec
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args.qubits)
        print(json.dumps(out), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    """The reference's own CUDA library replaying src/circuit.rs on a depth-bounded sample of the same circuit.
    The gate phase (one launch sequence per gate, cost independent of depth) and the density / seed phase (a fixed
    16 densities whatever the depth) are timed separately with CUDA events on the library's stream, and the
    full-depth step is  T_gates * (gates_full / gates_sampled) + T_densities  -- the sample's own ratio of gates to
    densities (31 : 16 at depth 2) is not the workload's (1550 : 16) and would understate the reference."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_replay as rr
    import torch
    torch.cuda.set_device(0)
    n = args.qubits
    dtype = np.complex64 if args.precision == "f32" else np.complex128
    if not rr.ref_available(args.precision, big=n > 30):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref not built (make -C oracle)"}))
        return
    depth = args.ref_depth
    circ = rr.RefCircuit(n, args.precision)
    n_gates, n_dens = build_brickwork(circ, n, depth)
    n_gates_full = len(brickwork_program(n, args.depth)[0])
    var, cts = brickwork_inputs(n, depth, dtype)
    cts_conj = [c.conj() for c in cts]
    marks = []

    def on_phase(name):          # the library runs on the legacy default stream, as torch's current stream does
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append((name, ev))

    def step():
        dens = circ.forward([], var)
        return dens, circ.backward(cts_conj, [], var)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    circ.on_phase = on_phase
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    ev0.record()
    on_phase("start")
    for _ in range(args.steps):
        dens, grads = step()
    on_phase("end")
    ev1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    dev_ms = ev0.elapsed_time(ev1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dens, grads)
    phase_ms = {"gates": 0.0, "densities": 0.0}
    for (name, a), (_, b) in zip(marks[:-1], marks[1:]):
        if name in phase_ms:
            phase_ms[name] += a.elapsed_time(b)
    t_gates, t_dens = phase_ms["gates"] / args.steps, phase_ms["densities"] / args.steps
    full_ms = t_gates * n_gates_full / n_gates + t_dens
    value = n_gates_full / (full_ms * 1e-3)
    host_overhead = wall / (dev_ms * 1e-3)
    sample = (f"reference CUDA library ({os.path.basename(circ.lib.path)}) replaying src/circuit.rs on "
              f"brickwork-{n}q depth {depth} of {args.depth} ({n_gates} gates + {n_dens} densities per sampled step), "
              f"one B200; gate phase {t_gates:.1f} ms, density + seed phase {t_dens:.1f} ms per sampled step; "
              f"full-depth step = gate phase x {n_gates_full}/{n_gates} + density phase = {full_ms:.0f} ms")
    out = {
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.precision,
        "data": "synthetic", "full_state_gate_applies_per_s": round(value, 3),
        "config": {"workload": f"brickwork-{n}q-depth{args.depth}-{args.precision}", "qubits": n, "depth": args.depth,
                   "gates": n_gates_full, "densities": n_dens, "depth_sampled": depth, "gates_sampled": n_gates,
                   "same_config": True,
                   "extrapolation": "value = gates(depth %d) / (T_gate_phase(depth %d) * gates_full / gates_sampled + "
                                    "T_density_phase); the reference's cost per gate does not depend on depth"
                                    % (args.depth, depth),
                   "sampled_step_ms": round(dev_ms / args.steps, 3), "extrapolated_full_step_ms": round(full_ms, 1),
                   "raw_sample_gate_applies_per_s": round(n_gates * args.steps / (dev_ms * 1e-3), 3)},
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": 0, "kind": "reference",
                         "sample": sample + " -- the reference has no CPU implementation; this is its own GPU code"},
        "e2e": {"value": round(value / host_overhead, 3), "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2,
                    help="timed steps of the workload; the secondary workloads (--secondary) run fixed counts: "
                         "VQSE-28 5 steps, 32 q f64 1 step")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--qubits", type=int, default=32, help="LOCAL qubits per GPU (total = qubits + log2(gpus))")
    ap.add_argument("--depth", type=int, default=100, help="brickwork layers / VQSE (ZZ, X) layer pairs")
    ap.add_argument("--workload", default="brickwork", choices=["brickwork", "vqse"])
    ap.add_argument("--ref-depth", type=int, default=2, help="depth of the bounded sample the reference arm runs")
    ap.add_argument("--precision", default="f32", choices=["f32", "f64"])
    ap.add_argument("--fuse", type=int, default=2, help="0: one pass per gate, 1: tiled passes, 2: register-blocked tiled passes")
    ap.add_argument("--tile-bits", type=int, default=0, help="T of the tiled passes (0: library default)")
    ap.add_argument("--low-bits", type=int, default=0, help="L lowest positions forced into every tile (0: default)")
    ap.add_argument("--max-tile-gates", type=int, default=0)
    ap.add_argument("--peer", type=int, default=1, help="sharded: 1 peer-memory swap kernel, 0 NCCL send/recv")
    ap.add_argument("--soa", type=int, default=1, help="f32 tile kernels: 1 pair-lane smem layout, 0 interleaved layout")
    ap.add_argument("--fusion", type=int, default=0, help="1: FusedCircuit (host-side gate fusion + gradient chain rule)")
    ap.add_argument("--rb-policy", type=int, default=-1, help="fuse=2 forward: 0 never register-block, 1 always, 2 by gate mix (default)")
    ap.add_argument("--batch-dens", type=int, default=-1, help="0: one sweep per density / seed")
    ap.add_argument("--tile-strategy", type=int, default=-1, help="scheduler tiling: 2 window growth with look-ahead (default), 1 window growth, 0 first-fit")
    ap.add_argument("--tc-rev", type=int, default=-1, help="f32 + tc: 1 fused one-sweep reverse step of a block (4*S), 0 three sweeps (6*S)")
    ap.add_argument("--tc-products", type=int, default=0, help="f32 + tc: 8 or 6 bf16 slice products per block (0: library default)")
    ap.add_argument("--tc", type=int, default=-1, help="f32: 1 tensor-core fused 6-qubit blocks, 0 FP32-pipe tile kernels only (-1: library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-check", action="store_true", help="skip the parity check that precedes the timed steps")
    ap.add_argument("--secondary", type=int, default=1,
                    help="1: after the default 32 q f32 run also measure VQSE-28 f32 and brickwork 32 q f64 (N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the densities and gradients of the last timed step of the workload (not of the "
                         "secondary workloads; with --impl reference, of its depth-bounded sample) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
