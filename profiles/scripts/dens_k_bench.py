"""Device time of the k-qubit density sweep (k_dens_k + its fixed-order final sum) and of the seed sweep (k_seed_k)
on states larger than L2: k = 3..6, positions low / high / mixed, 30 and 32 qubits f32 and 30 qubits f64.

Times come from the executor's CUDA-event profile (option "profile": events around each launch group on the
executing stream), after one warm-up call per shape; the median of REPS calls is reported.
  * density: forward() of a circuit holding one differentiable k-density (one density sweep, 1*S algorithmic bytes);
  * seed, created: backward() of that circuit (no adjoint yet: reads fwd, writes bwd, 2*S);
  * seed, accumulated: backward() of a circuit with two k-densities at the same program point minus the first
    (the second seed reads fwd and bwd and writes bwd, 3*S).
Each is also given as effective GB/s over the algorithmic bytes and as a multiple of one read of the state at the
measured copy peak of DESIGN.md section 6 (6452.8 GB/s).

    python profiles/scripts/dens_k_bench.py [--out FILE] [--reps 5] [--configs 30:f32,32:f32,30:f64]
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
COPY_PEAK_GBS = 6452.8


def positions(kind, n, k):
    if kind == "low":
        return list(range(k - 1, -1, -1))
    if kind == "high":
        return list(range(n - 1, n - 1 - k, -1))
    out = []                       # mixed: top and bottom qubits alternating, unsorted
    for j in range(k):
        out.append(n - 1 - j // 2 if j % 2 == 0 else j // 2)
    return out


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return name, q


def time_case(pkg, n, precision, pos, reps):
    dtype = np.complex64 if precision == "f32" else np.complex128
    d = 1 << len(pos)
    ct = (np.random.default_rng(0).normal(size=(d, d)) * (1 + 1j)).astype(dtype)
    res = {}
    for ndens in (1, 2):
        c = pkg.Circuit(n, precision=precision)
        c.set_option("profile", 1)
        for _ in range(ndens):
            c.get_dens_op_with_grad(pos)
        dens_ms, seed_ms = [], []
        for r in range(reps + 1):            # the first call warms up the shapes
            c.forward([], [])
            p = c.last_profile()
            c.backward([ct] * ndens, [], [])
            s = c.last_profile()
            if r:
                dens_ms.append(p["density"]["ms"] / p["density"]["launches"])
                seed_ms.append(s["seed"]["ms"])
        del c
        res[ndens] = (float(np.median(dens_ms)), float(np.median(seed_ms)))
    return res[1][0], res[1][1], res[2][1] - res[1][1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--configs", default="30:f32,32:f32,30:f64")
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
            for kind in ("low", "high", "mixed"):
                pos = positions(kind, n, k)
                dens, seed_new, seed_acc = time_case(pkg, n, precision, pos, args.reps)
                rec = {"n": n, "precision": precision, "k": k, "positions": kind, "pos": pos,
                       "density_ms": round(dens, 3), "density_gbs": round(S / dens / 1e6, 1),
                       "density_x_one_read": round(dens / one_read_ms, 2),
                       "seed_create_ms": round(seed_new, 3), "seed_create_gbs": round(2 * S / seed_new / 1e6, 1),
                       "seed_accumulate_ms": round(seed_acc, 3),
                       "seed_accumulate_gbs": round(3 * S / seed_acc / 1e6, 1),
                       "seed_accumulate_x_one_read": round(seed_acc / one_read_ms, 2)}
                lines.append(rec)
                print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
