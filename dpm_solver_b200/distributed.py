"""Multi-GPU: batch sharding with ONE broadcast of the scalar plan and no pixel traffic.

The solver path has no reduction across the batch (dynamic thresholding reduces inside a sample,
dpm_solver_pytorch.py:422), so rank r simply owns samples [r*B/W, (r+1)*B/W) -- the reference's own
multi-GPU story is one replica per GPU on disjoint batches (examples/ddpm_and_guided-diffusion/
main.py:249-265). The only thing that must agree between ranks is the per-step scalars; rank 0
broadcasts the packed coefficient plan once per run (a few hundred bytes over NCCL/NVLink, or gloo
in the CPU tests) so that every rank applies bit-identical fp32 coefficients. x, eps and the
buffered model values never leave their GPU.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch
import torch.distributed as dist

from .plan import Coeffs

_FLOAT_FIELDS = ("a", "c0", "c1", "c2", "w0", "w1", "w2", "w3", "w4", "cn")
_INT_FIELDS = ("form", "c0_on_old", "order", "r_tensor")
_WIDTH = len(_FLOAT_FIELDS) + len(_INT_FIELDS)


def shard_bounds(batch: int, rank: int, world: int):
    """Contiguous split of dim 0; the first (batch % world) ranks take one extra sample."""
    base, extra = divmod(batch, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_batch(x: torch.Tensor, rank: Optional[int] = None, world: Optional[int] = None) -> torch.Tensor:
    rank = dist.get_rank() if rank is None else rank
    world = dist.get_world_size() if world is None else world
    lo, hi = shard_bounds(x.shape[0], rank, world)
    return x[lo:hi]


def pack_plan(plan: Sequence[Coeffs]) -> torch.Tensor:
    """[len(plan), 14] float64 table (fp32 values and small ints are exact in float64)."""
    t = torch.zeros(len(plan), _WIDTH, dtype=torch.float64)
    for i, c in enumerate(plan):
        for j, f in enumerate(_FLOAT_FIELDS):
            t[i, j] = getattr(c, f)
        for j, f in enumerate(_INT_FIELDS):
            t[i, len(_FLOAT_FIELDS) + j] = float(int(getattr(c, f)))
    return t


def unpack_plan(t: torch.Tensor) -> List[Coeffs]:
    out = []
    for row in t.tolist():
        kw = {f: row[j] for j, f in enumerate(_FLOAT_FIELDS)}
        form, c0_on_old, order, r_tensor = (int(v) for v in row[len(_FLOAT_FIELDS):])
        out.append(Coeffs(form=form, c0_on_old=bool(c0_on_old), order=order, r_tensor=r_tensor, **kw))
    return out


def broadcast_plan(plan: Sequence[Coeffs], src: int = 0, group=None, device=None) -> List[Coeffs]:
    """Rank `src`'s plan on every rank: exactly one collective, len(plan)*14*8 bytes."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return list(plan)
    t = pack_plan(plan)
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else "cpu"
    t = t.to(device)
    dist.broadcast(t, src=src, group=group)
    return unpack_plan(t.cpu())
