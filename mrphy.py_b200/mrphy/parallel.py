r"""Spin sharding over the GPUs of one box (one process per GPU, ``torch.distributed``/NCCL).

Spins never interact (sims.py:91-126 is elementwise over `(N,*Nd)`); the only cross-spin operation of
forward+backward is the sum over spins that produces ``rf.grad``/``gr.grad`` (autograd of
beffective.py:137-165).  So each rank owns a contiguous range of the COMPACT spin axis ``nM`` with its
``loc_, Δf_, b1Map_, T1_, T2_, γ_, M_``; the waveform is replicated and the single collective is one
all-reduce(sum) of the flat ``[rf.grad ‖ gr.grad ‖ extras]`` buffer (N·nT·(2·nCoils+3) elements, 80 KB
for nT=4000).  Geometry stays global: the shard is a ``SpinArray`` with explicit ``loc_`` sliced from the
global cube -- do not rebuild a smaller ``SpinCube`` (``_update_loc_`` centres on ``n//2``).

Per-spin gradients (``loc_``, ``Δf_``, ``b1Map_``, ``γ_`` requiring grad) are local to a shard and need no collective.
A ``Δf`` or ``γ`` that is ONE tensor broadcast over spins gets, on each rank, only the sum over that rank's spins; this
module does not all-reduce it -- sum it over ranks yourself if you need the global gradient.
"""
from typing import Optional, Tuple

import torch
import torch.distributed as dist
from torch import Tensor

from mrphy import mobjs

__all__ = ['shard_range', 'shard_spins', 'shard_batch', 'allreduce_waveform_grads', 'flat_wave_grads']


def shard_range(nM: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced split of ``range(nM)``: the first ``nM % world`` ranks get one extra spin."""
    base, extra = divmod(nM, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_spins(obj, rank: int, world: int, *, loc_: Optional[Tensor] = None, Δf_: Optional[Tensor] = None,
                b1Map_: Optional[Tensor] = None, device: Optional[torch.device] = None):
    """Rank ``rank``'s slab of a ``SpinCube``/``SpinArray``.

    Returns ``(spinarray, kw)``: a compact all-True-mask ``SpinArray`` of shape `(N, nLocal)` and the keyword
    arguments (``loc_``, ``Δf_``, ``b1Map_``) to pass to ``spinarray.applypulse(pulse, **kw)``.
    """
    sp = obj.spinarray if isinstance(obj, mobjs.SpinCube) else obj
    lo, hi = shard_range(sp.nM, rank, world)
    device = sp.device if device is None else device
    if isinstance(obj, mobjs.SpinCube):
        loc_ = obj.loc_ if loc_ is None else loc_
        Δf_ = obj.Δf_ if Δf_ is None else Δf_
    assert loc_ is not None, 'a SpinArray has no geometry: pass loc_'
    cut = lambda x: None if x is None else (x[:, lo:hi] if x.shape[1] != 1 else x).to(device)
    local = mobjs.SpinArray((sp.shape[0], hi - lo), T1_=cut(sp.T1_), T2_=cut(sp.T2_), γ_=cut(sp.γ_),
                            M_=cut(sp.M_).contiguous(), device=device, dtype=sp.dtype)
    return local, {'loc_': cut(loc_).contiguous(), 'Δf_': cut(Δf_), 'b1Map_': cut(b1Map_)}


def shard_batch(obj, pulse, rank: int, world: int, *, loc_: Optional[Tensor] = None, Δf_: Optional[Tensor] = None,
                b1Map_: Optional[Tensor] = None, device: Optional[torch.device] = None):
    """The batch axis ``N`` as the shard axis (the second natural one: N different pulses on N copies of the spins, e.g. 64
    candidate pulses): rank ``rank`` gets the entries ``[lo, hi)`` of the spins AND of the pulse.  Every entry's ``rf.grad`` /
    ``gr.grad`` is complete on the rank that owns it, so this split needs NO collective at all.

    Returns ``(spinarray, kw, pulse_local, (lo, hi))``; quantities with a broadcast batch dimension (size 1) are shared.
    The local pulse holds views ``pulse.rf[lo:hi]``, ``pulse.gr[lo:hi]``: gradients reach the caller's leaves through them.
    """
    sp = obj.spinarray if isinstance(obj, mobjs.SpinCube) else obj
    N = sp.shape[0]
    assert pulse.rf.shape[0] == N, 'pulse and spins disagree on the batch size'
    lo, hi = shard_range(N, rank, world)
    device = sp.device if device is None else device
    if isinstance(obj, mobjs.SpinCube):
        loc_ = obj.loc_ if loc_ is None else loc_
        Δf_ = obj.Δf_ if Δf_ is None else Δf_
    assert loc_ is not None, 'a SpinArray has no geometry: pass loc_'

    def cut(x):
        if x is None or not isinstance(x, Tensor):
            return x
        return (x[lo:hi] if (x.ndim >= 1 and x.shape[0] == N and N > 1) else x).to(device)

    local = mobjs.SpinArray((hi - lo, sp.nM), T1_=cut(sp.T1_), T2_=cut(sp.T2_), γ_=cut(sp.γ_), M_=cut(sp.M_).contiguous(),
                            device=device, dtype=sp.dtype)
    p_local = mobjs.Pulse(rf=cut(pulse.rf), gr=cut(pulse.gr), dt=cut(pulse.dt), gmax=cut(pulse.gmax), smax=cut(pulse.smax),
                          rfmax=cut(pulse.rfmax), desc=pulse.desc, device=device, dtype=pulse.dtype)
    return local, {'loc_': cut(loc_).contiguous(), 'Δf_': cut(Δf_), 'b1Map_': cut(b1Map_)}, p_local, (lo, hi)


def flat_wave_grads(rf: Tensor, gr: Tensor) -> Optional[Tensor]:
    """The fused backward writes ``rf.grad`` and ``gr.grad`` into ONE buffer ``[rf.grad | gr.grad | GRAD_TAIL spare]``
    (``mrphy._ops``); autograd hands both views to the leaves unchanged.  Returns that buffer as a 1-D tensor, or None
    when the gradients are separate tensors (accumulated over several backward calls, produced by other operators...)."""
    from mrphy import _ops
    a, b = rf.grad, gr.grad
    if a is None or b is None or a.dtype != b.dtype or not (a.is_contiguous() and b.is_contiguous()):
        return None
    sa = a.untyped_storage()
    if sa.data_ptr() != b.untyped_storage().data_ptr() or b.storage_offset() != a.storage_offset() + a.numel():
        return None
    n = a.numel() + b.numel() + _ops.GRAD_TAIL
    if (a.storage_offset() + n) * a.element_size() > sa.nbytes():
        return None
    return torch.empty(0, dtype=a.dtype, device=a.device).set_(sa, a.storage_offset(), (n,), (1,))


def allreduce_waveform_grads(rf: Tensor, gr: Tensor, *extras: Tensor, group=None) -> None:
    """Sum ``rf.grad``, ``gr.grad`` (and any extra tensors, e.g. the scalar loss) over ranks, in place, with ONE
    all-reduce.  After a fused backward the gradients already live in one flat buffer: the extras (up to GRAD_TAIL
    elements) ride in its spare tail and the collective runs in place on it -- no gather, no scatter; captured into a
    CUDA graph with the step it costs no launch of its own.  Otherwise the parts are concatenated and copied back."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return
    from mrphy import _ops
    flat = flat_wave_grads(rf, gr)
    if flat is not None and sum(e.numel() for e in extras) <= _ops.GRAD_TAIL:
        off = flat.numel() - _ops.GRAD_TAIL
        slots = []
        for e in extras:
            slots.append(flat[off:off + e.numel()])
            slots[-1].copy_(e.reshape(-1))
            off += e.numel()
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        for e, sl in zip(extras, slots):
            e.copy_(sl.reshape(e.shape))
        return
    parts = [rf.grad, gr.grad, *extras]
    flat = torch.cat([p.reshape(-1) for p in parts])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    off = 0
    for p in parts:
        n = p.numel()
        p.copy_(flat[off:off + n].reshape(p.shape))
        off += n
