"""Domain decomposition of ONE model over several GPUs (SURVEY.md 8e-ii, BASELINE configs[4]).

One process per GPU (torchrun).  Every rank builds a `TransportBackend` with `dd_rank` / `dd_world` set on
the whole mesh; the library cuts the rows into `world` strips across the flow, and the ranks exchange
boundary rows and BiCGSTAB dot products directly over NVLink peer memory from inside the kernels
(csrc/cwr_kernels.cuh: peer_ptr, k_halo_push, dd_allreduce, the halo barrier of k_precond_gs).  The only
thing the host exchanges is the CUDA IPC handle of each rank's slab, once, through `torch.distributed` --
plumbing, not data path.  This module is that plumbing plus the merge of the per-rank outputs.
"""
from __future__ import annotations

from typing import Optional

import numpy as np

from .backend import IPC_HANDLE_BYTES, TransportBackend


def exchange_ipc_handles(local: bytes, rank: int, world: int, group=None, device: Optional[str] = None) -> bytes:
    """All-gather of the 64-byte CUDA IPC handles in rank order (uint8 tensor on `device` for NCCL, CPU for gloo)."""
    import torch
    import torch.distributed as dist
    assert len(local) == IPC_HANDLE_BYTES
    if world == 1:
        return local
    if device is None:
        device = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    mine = torch.tensor(list(local), dtype=torch.uint8, device=device)
    out = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(out, mine, group=group)
    return b"".join(bytes(t.cpu().tolist()) for t in out)


def merge_owned(local: np.ndarray, owned: np.ndarray, axis: int = -1, group=None, device: Optional[str] = None) -> np.ndarray:
    """Every rank holds `local` valid where `owned` (a partition over the ranks): sum of the masked arrays =
    the whole array on every rank.  (Outputs only: the solver itself never goes through the host.)"""
    import torch
    import torch.distributed as dist
    mask = np.expand_dims(owned, tuple(i for i in range(local.ndim) if i != axis % local.ndim)) if local.ndim > 1 else owned
    part = np.where(mask, local, 0.0)
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return part
    if device is None:
        device = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
    t = torch.from_numpy(np.ascontiguousarray(part)).to(device)
    dist.all_reduce(t, group=group)
    return t.cpu().numpy()


class DomainDecomposedBackend(TransportBackend):
    """A TransportBackend that owns one strip of the mesh; same calls as the single-GPU backend, made by
    every rank in the same order with the same arguments.  `attach()` after construction (collective)."""

    def __init__(self, f1, f2, n_face, n_time, n_constituents, diffusion_coefficient, rank: int, world: int,
                 device: int = 0, group=None, flow_hint=None, **options):
        options.setdefault("solver_path", 1)
        super().__init__(f1, f2, n_face, n_time, n_constituents, diffusion_coefficient, device=device,
                         flow_hint=flow_hint, dd_rank=rank, dd_world=world, **options)
        self.rank, self.world, self.group = rank, world, group
        self._owned_cells = self._owned_edges = None

    def attach(self):
        """Collective: map every peer's slab (call after the hydrodynamics are uploaded, so that the strips
        are already aligned with the flow, and before the first step)."""
        handles = exchange_ipc_handles(self.dd_export(), self.rank, self.world, self.group)
        self.dd_attach(handles)
        self.info, self._owned_cells, self._owned_edges = self.dd_layout()
        import torch.distributed as dist
        if dist.is_initialized():        # no rank steps (and stores into a peer's slab) before every rank has mapped it
            dist.barrier(group=self.group)
        return self.info

    # -- merged outputs (collective) ---------------------------------------------------------------
    def gather_state_all(self, t: int) -> np.ndarray:
        """(K, n) concentrations of all real cells at time index t, on every rank."""
        return merge_owned(self.get_state_all(t), self._owned_cells, axis=1, group=self.group)

    def gather_mass_totals(self, k: int, t_start: int, t_end: int):
        m = self.mass_totals(k, t_start, t_end)
        v = merge_owned(np.array([m.vol_start, m.mass_start, m.vol_end, m.mass_end]), np.ones(4, bool), group=self.group)
        return tuple(float(x) for x in v)

    def gather_reaction_mass(self, k: int) -> float:
        """Reaction mass of constituent k over the whole mesh: the sum of the ranks' partial sums."""
        v = merge_owned(np.array([self.reaction_mass(k)]), np.ones(1, bool), group=self.group)
        return float(v[0])
