"""`AutoGradCircuit`: Python wrapper with reverse-mode differentiation, mirror
of /root/reference/src/qdc/circuit.py:8-202 (same builder methods, same
`build() -> (simple_run, autodiff_run)` contract, argument order
`(var_gates, const_gates)` at this level vs `(const, var)` one level down).

The reference glues `Circuit.forward/backward` into JAX with `jax.custom_vjp`
(src/qdc/circuit.py:177-201).  JAX is optional here:
  * if `jax` is importable, `autodiff_run` is the same `custom_vjp` function;
  * otherwise `autodiff_run` accepts torch tensors (differentiable through
    `torch.autograd`) or NumPy arrays (forward only), and exposes
    `autodiff_run.vjp(var_gates, const_gates, density_cotangents)` which is the
    reference's `bwd_run` (cotangents are conjugated, src/qdc/circuit.py:193).
Cotangent convention: JAX's.  The returned gate gradients g satisfy
dL = Re sum(g * dU)  (src/test_autodiff.py:159-164).
"""
from __future__ import annotations

from typing import Callable, List, Tuple

import numpy as np

from ..quantum_differentiable_circuit import Circuit

try:  # pragma: no cover - jax is not part of this image
    import jax  # type: ignore
    from jax import custom_vjp  # type: ignore
    _HAVE_JAX = True
except Exception:  # noqa: BLE001
    _HAVE_JAX = False


def _np(x, dtype):
    """np.asarray() of a JAX / torch / NumPy array (src/qdc/circuit.py:173-174)."""
    if hasattr(x, "detach"):
        x = x.detach().cpu().numpy()
    a = np.asarray(x)
    return a if a.dtype == dtype else a.astype(dtype)


class _AutodiffRun:
    """Callable returned as `autodiff_run` when JAX is absent."""

    def __init__(self, circuit: Circuit):
        self._c = circuit

    def forward(self, var_gates, const_gates) -> List[np.ndarray]:
        dt = self._c.dtype
        return self._c.forward([_np(g, dt) for g in const_gates], [_np(g, dt) for g in var_gates])

    def vjp(self, var_gates, const_gates, density_cotangents) -> List[np.ndarray]:
        """`bwd_run` of src/qdc/circuit.py:190-197 (must follow `forward`)."""
        dt = self._c.dtype
        return self._c.backward(
            [_np(g, dt).conj() for g in density_cotangents],
            [_np(g, dt) for g in const_gates],
            [_np(g, dt) for g in var_gates],
        )

    def __call__(self, var_gates, const_gates):
        try:
            import torch
        except Exception:  # noqa: BLE001
            torch = None
        if torch is not None and any(isinstance(g, torch.Tensor) for g in list(var_gates) + list(const_gates)):
            return _torch_apply(self, list(var_gates), list(const_gates))
        return self.forward(var_gates, const_gates)


def _torch_gather(tensors, np_dtype):
    """All gate tensors -> NumPy with ONE device-to-host transfer (SURVEY.md 8(f) item 3; the
    reference converts gate by gate, src/qdc/circuit.py:173-195, i.e. one blocking copy per gate
    when the parameters live on the GPU)."""
    import torch
    if not tensors:
        return []
    tdt = torch.complex64 if np_dtype == np.complex64 else torch.complex128
    flat = torch.cat([t.detach().reshape(-1).to(tdt) for t in tensors])
    host = flat.cpu().numpy()
    out, o = [], 0
    for t in tensors:
        out.append(host[o:o + t.numel()].reshape(tuple(t.shape)))
        o += t.numel()
    return out


def _torch_scatter(arrays, like):
    """NumPy results -> tensors on the device / dtype of `like` with ONE host-to-device transfer."""
    import torch
    if not arrays:
        return []
    flat = torch.from_numpy(np.concatenate([np.ascontiguousarray(a).reshape(-1) for a in arrays]))
    flat = flat.to(device=like[0].device)
    out, o = [], 0
    for a, t in zip(arrays, like):
        out.append(flat[o:o + a.size].reshape(tuple(t.shape)).to(t.dtype))
        o += a.size
    return out


def _torch_apply(run: _AutodiffRun, var_gates, const_gates):
    import torch

    n_var = len(var_gates)
    as_t = lambda g: g if isinstance(g, torch.Tensor) else torch.as_tensor(np.asarray(g))  # noqa: E731
    var_gates, const_gates = [as_t(g) for g in var_gates], [as_t(g) for g in const_gates]
    dt = run._c.dtype
    dev = next((g.device for g in var_gates + const_gates if g.is_cuda), torch.device("cpu"))

    class _Fn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, *gates):
            host = _torch_gather(list(gates), dt)     # one D2H for every gate of the circuit
            ctx.host_gates = host
            dens = run._c.forward(host[n_var:], host[:n_var])
            flat = torch.from_numpy(np.concatenate([d.reshape(-1) for d in dens]) if dens else np.zeros(0, dt))
            flat = flat.to(dev)                       # one H2D for every density
            out, o = [], 0
            for d in dens:
                out.append(flat[o:o + d.size].reshape(d.shape))
                o += d.size
            ctx.var_like = gates[:n_var]
            return tuple(out)

        @staticmethod
        def backward(ctx, *grad_outputs):
            host = ctx.host_gates
            # torch's complex gradient is the conjugate of the JAX cotangent; Circuit.backward wants the
            # conjugated JAX cotangent (src/qdc/circuit.py:193), i.e. torch's gradient as it is
            cts = _torch_gather(list(grad_outputs), dt)
            grads = run._c.backward(cts, host[n_var:], host[:n_var])
            out = _torch_scatter([g.conj() for g in grads], ctx.var_like)
            return tuple(out) + (None,) * (len(host) - n_var)

    return list(_Fn.apply(*var_gates, *const_gates))


class AutoGradCircuit:

    def __init__(self, qubits_number: int, precision: str | None = None, fused: bool = False):
        """Quantum circuit with automatic differentiation (src/qdc/circuit.py:10-12).  `fused=True` puts
        host-side gate fusion in front of the executor (fusion.py; opt-in, not in the reference)."""
        if fused:
            from ..fusion import FusedCircuit
            self.circuit = FusedCircuit(qubits_number, precision=precision)
        else:
            self.circuit = Circuit(qubits_number, precision=precision)

    def set_state_from_vector(self, vec):
        """Set initial state from an array (src/qdc/circuit.py:14-22)."""
        self.circuit.set_state_from_vector(_np(vec, self.circuit.dtype))

    # 1:1 forwarding builders, src/qdc/circuit.py:24-158.  Qubits are enumerated
    # starting from the innermost one; pos2 is the 'control', pos1 the 'target'.
    def add_q2_const_gate(self, pos2: int, pos1: int): self.circuit.add_q2_const_gate(pos2, pos1)
    def add_q2_const_gate_nonu(self, pos2: int, pos1: int): self.circuit.add_q2_const_gate_nonu(pos2, pos1)
    def add_q2_const_gate_diag(self, pos2: int, pos1: int): self.circuit.add_q2_const_gate_diag(pos2, pos1)
    def add_q2_var_gate(self, pos2: int, pos1: int): self.circuit.add_q2_var_gate(pos2, pos1)
    def add_q2_var_gate_nonu(self, pos2: int, pos1: int): self.circuit.add_q2_var_gate_nonu(pos2, pos1)
    def add_q2_var_gate_diag(self, pos2: int, pos1: int): self.circuit.add_q2_var_gate_diag(pos2, pos1)
    def add_q1_const_gate(self, pos: int): self.circuit.add_q1_const_gate(pos)
    def add_q1_const_gate_nonu(self, pos: int): self.circuit.add_q1_const_gate_nonu(pos)
    def add_q1_var_gate(self, pos: int): self.circuit.add_q1_var_gate(pos)
    def add_q1_var_gate_nonu(self, pos: int): self.circuit.add_q1_var_gate_nonu(pos)
    def get_q2_dens_op(self, pos2: int, pos1: int): self.circuit.get_q2_dens_op(pos2, pos1)
    def get_q1_dens_op(self, pos: int): self.circuit.get_q1_dens_op(pos)
    def get_q2_dens_op_with_grad(self, pos2: int, pos1: int): self.circuit.get_q2_dens_op_with_grad(pos2, pos1)
    def get_q1_dens_op_with_grad(self, pos: int): self.circuit.get_q1_dens_op_with_grad(pos)
    # densities on 1..6 qubits, positions[0] the most significant bit (Circuit.get_dens_op)
    def get_dens_op(self, positions): self.circuit.get_dens_op(positions)
    def get_dens_op_with_grad(self, positions): self.circuit.get_dens_op_with_grad(positions)
    # gates on 1..6 qubits, positions[0] the most significant bit (Circuit.add_const_gate)
    def add_const_gate(self, positions): self.circuit.add_const_gate(positions)
    def add_var_gate(self, positions): self.circuit.add_var_gate(positions)
    def add_const_gate_nonu(self, positions): self.circuit.add_const_gate_nonu(positions)
    def add_var_gate_nonu(self, positions): self.circuit.add_var_gate_nonu(positions)
    # diagonal gates on 1..6 qubits, positions[0] the most significant bit (Circuit.add_const_gate_diag)
    def add_const_gate_diag(self, positions): self.circuit.add_const_gate_diag(positions)
    def add_var_gate_diag(self, positions): self.circuit.add_var_gate_diag(positions)
    def add_const_gate_diag_nonu(self, positions): self.circuit.add_const_gate_diag_nonu(positions)
    def add_var_gate_diag_nonu(self, positions): self.circuit.add_var_gate_diag_nonu(positions)

    def build(self) -> Tuple[Callable, Callable]:
        """Returns (simple_run, autodiff_run), src/qdc/circuit.py:160-202.

        simple_run(var_gates, const_gates) evaluates every requested density
        matrix and has no backward pass; autodiff_run evaluates only those with
        gradient and supports the backward pass."""
        dt = self.circuit.dtype

        def simple_run(var_gates, const_gates):
            return self.circuit.run([_np(g, dt) for g in const_gates], [_np(g, dt) for g in var_gates])

        if not _HAVE_JAX:
            return simple_run, _AutodiffRun(self.circuit)

        @custom_vjp
        def autodiff_run(var_gates, const_gates):  # pragma: no cover
            return self.circuit.forward([_np(g, dt) for g in const_gates], [_np(g, dt) for g in var_gates])

        def fwd_run(var_gates, const_gates):  # pragma: no cover
            dens = self.circuit.forward([_np(g, dt) for g in const_gates], [_np(g, dt) for g in var_gates])
            return dens, (const_gates, var_gates)

        def bwd_run(res, density_grads):  # pragma: no cover
            const_gates, var_gates = res
            grads = self.circuit.backward(
                [_np(g, dt).conj() for g in density_grads],
                [_np(g, dt) for g in const_gates],
                [_np(g, dt) for g in var_gates],
            )
            return grads, None

        autodiff_run.defvjp(fwd_run, bwd_run)
        return simple_run, autodiff_run
