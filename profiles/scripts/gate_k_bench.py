"""Device time of the k-qubit gate sweeps on states larger than L2: the apply sweep (k_gate_k, forward pass) and the
fused reverse step of a variable gate (k_gate_k_rev + the fixed-order gradient sum), k = 3..6, positions low and high,
32 and 30 qubits f32 and 30 qubits f64.

Times come from the executor's CUDA-event profile (option "profile": events around each launch group on the
executing stream), after one warm-up call per shape; the median of REPS calls is reported.  The circuit is one
variable k-qubit gate followed by a differentiable one-qubit density (whose sweeps are profiled separately):
  * apply: forward() of that circuit, category gate_k_fwd (reads and writes the state, 2*S algorithmic bytes);
  * reverse: backward() of it, category gate_k_rev (reads and writes the state and the adjoint, 4*S).
Each is also given as effective GB/s over the algorithmic bytes and as a multiple of one read of the state at the
measured copy peak of DESIGN.md section 6 (6452.8 GB/s).

    python profiles/scripts/gate_k_bench.py [--out FILE] [--reps 5] [--configs 32:f32,30:f32,30:f64]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "scripts"))
from dens_k_bench import COPY_PEAK_GBS, card, positions  # noqa: E402


def time_case(pkg, n, precision, pos, reps):
    dtype = np.complex64 if precision == "f32" else np.complex128
    d = 1 << len(pos)
    z = np.random.default_rng(0).normal(size=(d, d)) + 1j * np.random.default_rng(1).normal(size=(d, d))
    u = np.linalg.qr(z)[0].reshape(-1).astype(dtype)
    ct = np.eye(2, dtype=dtype)
    c = pkg.Circuit(n, precision=precision)
    c.set_option("profile", 1)
    c.add_var_gate(pos)
    c.get_q1_dens_op_with_grad(n // 2)
    apply_ms, rev_ms = [], []
    for r in range(reps + 1):            # the first call warms up the shapes
        c.forward([], [u])
        p = c.last_profile()
        c.backward([ct], [], [u])
        s = c.last_profile()
        if r:
            apply_ms.append(p["gate_k_fwd"]["ms"])
            rev_ms.append(s["gate_k_rev"]["ms"])
    del c
    return float(np.median(apply_ms)), float(np.median(rev_ms))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--configs", default="32:f32,30:f32,30:f64")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "needs a GPU"
    pkg = importlib.import_module("differentiable-quantum-circuit-cuda_b200")
    name, plimit = card()
    lines = [{"card": name, "power_limit": plimit, "copy_peak_gbs": COPY_PEAK_GBS, "reps": args.reps}]
    print(json.dumps(lines[0]), flush=True)
    for cfg in args.configs.split(","):
        n, precision = int(cfg.split(":")[0]), cfg.split(":")[1]
        S = (8 if precision == "f32" else 16) << n
        one_read_ms = S / (COPY_PEAK_GBS * 1e9) * 1e3
        for k in (3, 4, 5, 6):
            for kind in ("low", "high"):
                pos = positions(kind, n, k)
                apply_ms, rev_ms = time_case(pkg, n, precision, pos, args.reps)
                rec = {"n": n, "precision": precision, "k": k, "positions": kind, "pos": pos,
                       "apply_bytes": 2 * S, "apply_ms": round(apply_ms, 3),
                       "apply_gbs": round(2 * S / apply_ms / 1e6, 1),
                       "apply_x_one_read": round(apply_ms / one_read_ms, 2),
                       "reverse_bytes": 4 * S, "reverse_ms": round(rev_ms, 3),
                       "reverse_gbs": round(4 * S / rev_ms / 1e6, 1),
                       "reverse_x_one_read": round(rev_ms / one_read_ms, 2)}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
