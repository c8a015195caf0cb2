"""Device time of the diagonal k-qubit gate sweeps on states larger than L2, k = 1..6, positions low and high, 32 and
30 qubits f32 and 30 qubits f64, each next to the two yardsticks measured in the same run:
  * the diagonal: the apply sweep (k_diag_k, forward pass, category diag_k_fwd, 2*S) and the fused reverse step of a
    variable diagonal (k_diag_k_rev + the fixed-order gradient sum, category diag_k_rev, 4*S);
  * the two-qubit diagonal (option fuse = 0, so that it is not absorbed into a tile pass): fwd_diag / rev_diag, on the
    lowest two of the positions (k = 1: position and its neighbour), once per configuration and position class;
  * the dense k-qubit gate with U = diag(d) (add_var_gate; gate_k_fwd / gate_k_rev for k >= 3, fwd_q1 / rev_q1 and
    fwd_q2 / rev_q2 for k = 1, 2 under fuse = 0).
Times come from the executor's CUDA-event profile after one warm-up call per shape; the median of REPS calls is
reported.  The circuit is the gate followed by a differentiable one-qubit density (profiled separately).

    python profiles/scripts/diag_k_bench.py [--out FILE] [--reps 5] [--configs 32:f32,30:f32,30:f64]
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


def time_case(pkg, n, precision, add, gate, cats, reps):
    """median (apply ms, reverse ms) of the categories `cats` = (forward, reverse) for one variable gate"""
    dtype = np.complex64 if precision == "f32" else np.complex128
    c = pkg.Circuit(n, precision=precision)
    c.set_option("profile", 1)
    c.set_option("fuse", 0)
    add(c)
    c.get_q1_dens_op_with_grad(n // 2)
    g = np.asarray(gate, dtype=dtype)
    ct = np.eye(2, dtype=dtype)
    apply_ms, rev_ms = [], []
    for r in range(reps + 1):            # the first call warms up the shapes
        c.forward([], [g])
        p = c.last_profile()
        c.backward([ct], [], [g])
        s = c.last_profile()
        if r:
            apply_ms.append(p[cats[0]]["ms"])
            rev_ms.append(s[cats[1]]["ms"])
    del c
    return float(np.median(apply_ms)), float(np.median(rev_ms))


DENSE_CATS = {1: ("fwd_q1", "rev_q1"), 2: ("fwd_q2", "rev_q2")}


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
    rng = np.random.default_rng(0)
    for cfg in args.configs.split(","):
        n, precision = int(cfg.split(":")[0]), cfg.split(":")[1]
        S = (8 if precision == "f32" else 16) << n
        for kind in ("low", "high"):
            p2 = positions(kind, n, 2)
            d4 = np.exp(1j * rng.uniform(0, 6.3, size=4))
            q2a, q2r = time_case(pkg, n, precision, lambda c: c.add_q2_var_gate_diag(p2[0], p2[1]), d4,
                                 ("fwd_diag", "rev_diag"), args.reps)
            for k in range(1, 7):
                pos = positions(kind, n, k)
                d = np.exp(1j * rng.uniform(0, 6.3, size=1 << k))
                # (k = 2 unitary is the two-qubit diagonal itself: the NonU kind runs the new sweeps)
                add_d = (lambda c: c.add_var_gate_diag_nonu(pos)) if k == 2 else (lambda c: c.add_var_gate_diag(pos))
                da, dr = time_case(pkg, n, precision, add_d, d, ("diag_k_fwd", "diag_k_rev"), args.reps)
                ua, ur = time_case(pkg, n, precision, lambda c: c.add_var_gate(pos), np.diag(d).reshape(-1),
                                   DENSE_CATS.get(k, ("gate_k_fwd", "gate_k_rev")), args.reps)
                rec = {"n": n, "precision": precision, "k": k, "positions": kind, "pos": pos,
                       "apply_ms": round(da, 3), "apply_gbs": round(2 * S / da / 1e6, 1),
                       "reverse_ms": round(dr, 3), "reverse_gbs": round(4 * S / dr / 1e6, 1),
                       "q2diag_apply_ms": round(q2a, 3), "q2diag_reverse_ms": round(q2r, 3),
                       "apply_vs_q2diag": round(da / q2a, 3), "reverse_vs_q2diag": round(dr / q2r, 3),
                       "dense_apply_ms": round(ua, 3), "dense_reverse_ms": round(ur, 3),
                       "apply_speedup_vs_dense": round(ua / da, 2), "reverse_speedup_vs_dense": round(ur / dr, 2)}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
