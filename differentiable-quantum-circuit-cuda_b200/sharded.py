"""`ShardedCircuit`: the same `Circuit` surface over 2^g GPUs of one NVLink /
NVSwitch box, one process per GPU (torch.distributed for the plumbing).

The statevector is sharded by the top g global qubits; the C++ executor
(csrc/circuit.cuh) runs local passes and NCCL half-shard exchanges for qubit
remaps, and returns per-rank PARTIAL densities / gradients, which are summed
here with one small all-reduce per call.  No reference counterpart (the
reference links no communication library, /root/reference/build.rs:14-16).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from ._ffi import default_precision, get_lib
from .quantum_differentiable_circuit import Circuit


class ShardedCircuit(Circuit):
    def __init__(self, qubits_number: int, precision: str | None = None, group=None):
        import torch
        import torch.distributed as dist

        assert dist.is_initialized(), "ShardedCircuit needs torch.distributed (one process per GPU)"
        self._dist, self._torch, self._group = dist, torch, group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self._lib = get_lib(precision or default_precision())
        self.qubits_number = int(qubits_number)
        self.local_qubits = self.qubits_number - (self.world.bit_length() - 1)
        # bootstrap the NCCL communicator of the C++ executor
        uid = np.zeros(128, dtype=np.uint8)
        if self.rank == 0:
            self._lib.call("qdc_nccl_unique_id", uid.ctypes.data)
        t = torch.from_numpy(uid).cuda()
        dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        uid = t.cpu().numpy()
        h = C.c_void_p()
        self._lib.call("qdc_circuit_new_sharded", C.byref(h), self.qubits_number, self.rank, self.world,
                       uid.ctypes.data)
        self._h = h
        self._kinds = []
        self._dims = []

    @property
    def peer_exchange(self) -> bool:
        """True when remap exchanges run as the fused NVLink peer-memory swap kernel."""
        return bool(self._lib.cdll.qdc_circuit_peer_exchange(self._h))

    def _allreduce(self, arrays):
        if not arrays:
            return arrays
        flat = np.concatenate([a.reshape(-1) for a in arrays])
        # sum in double precision regardless of the build
        t = self._torch.from_numpy(flat.astype(np.complex128).view(np.float64)).cuda()
        self._dist.all_reduce(t, group=self._group)
        flat = t.cpu().numpy().view(np.complex128).astype(self._lib.cdtype)
        out, o = [], 0
        for a in arrays:
            out.append(flat[o:o + a.size].reshape(a.shape)); o += a.size
        return out

    def set_state_from_vector(self, vector):
        """`vector` is the FULL 2^n state (every rank passes the same array) or this
        rank's shard of 2^(n - g) entries."""
        v = self._lib.host(vector)
        shard = 1 << self.local_qubits
        if v.size == shard << (self.world.bit_length() - 1) and self.world > 1:
            v = np.ascontiguousarray(v[self.rank * shard:(self.rank + 1) * shard])
        self._lib.call("qdc_circuit_set_state_from_host", self._h, v.ctypes.data, v.size)

    def run(self, const_gates, var_gates):
        return self._allreduce(super().run(const_gates, var_gates))

    def forward(self, const_gates, var_gates):
        return self._allreduce(super().forward(const_gates, var_gates))

    def backward(self, grads_wrt_density, const_gates, var_gates):
        return self._allreduce(super().backward(grads_wrt_density, const_gates, var_gates))

    def save_state(self, path: str):
        """One file per rank: `path` with ".rank{r}of{w}" appended (state_io.assemble re-joins them)."""
        super().save_state(f"{path}.rank{self.rank}of{self.world}")

    def load_state(self, path: str):
        super().load_state(f"{path}.rank{self.rank}of{self.world}")

    def get_cpu_state_copy(self):
        """This rank's shard in the current physical layout (2^(n - g) entries)."""
        out = np.empty(1 << self.local_qubits, dtype=self._lib.cdtype)
        self._lib.call("qdc_circuit_copy_state_to_host", self._h, out.ctypes.data)
        return out
