r"""Bloch simulation with explicit Jacobian operations -- CUDA (sm_100a) implementation.

Public surface of the reference module (``/root/reference/mrphy/sims.py``): ``blochsim``,
``BlochSim``, ``freeprec``, ``FreePrec`` with the same argument shapes, dtypes and autograd
behaviour.  ``BlochSim`` stays a ``torch.autograd.Function`` with the reference signature
``forward(ctx, Mi, Beff, T1, T2, γ, dt)`` (sims.py:31-40) and
``backward(ctx, grad_Mo) -> (grad_Mi, grad_Beff, None, None, None, None)`` (sims.py:134-138,269),
but both directions are single CUDA kernels behind the C ABI (``mrphy_blochsim_beff_fwd/bwd``).

Differences a user can observe, all supersets: the per-step intermediates are not cached (10 floats per
spin-step upstream, sims.py:84-88), so memory is O(nM*nT/K); ``backward`` may be called more than once
(upstream mutates its saved tensors, sims.py:234-259); ``grad_Mi`` is also correct for per-spin ``γ``
(upstream indexing bug at sims.py:267).
"""
from typing import Optional, Tuple

import torch
from torch import Tensor
from torch.autograd import Function

from mrphy import γH, dt0, π  # noqa: F401
from mrphy import _cabi, _ops

__all__ = ['blochsim']


_flat_param = _ops.flat_param


class BlochSim(Function):
    r"""BlochSim with explicit Jacobian operation (backward).

    Only differentiable w.r.t. ``Mi`` and ``Beff`` (as upstream, sims.py:27).
    """

    @staticmethod
    def forward(ctx, Mi: Tensor, Beff: Tensor, T1: Optional[Tensor], T2: Optional[Tensor], γ: Tensor,
                dt: Tensor) -> Tensor:
        r"""Forward evolution.

        - ``Mi``: `(N, *Nd, xyz)`;  ``Beff``: `(N, *Nd, nT, xyz)` Gauss
        - ``T1``, ``T2``, ``γ``: `(N ⊻ 1, *Nd ⊻ 1.., 1, 1)`;  ``dt``: `(N ⊻ 1, 1.., 1, 1)`
        - returns ``Mo``: `(N, *Nd, xyz)`
        """
        _ops._require_cuda(Mi, Beff)
        assert (T1 is None) == (T2 is None)          # both or neither (sims.py:68)
        NNd, nT = Beff.shape[:-2], Beff.shape[-2]
        N, Nd = NNd[0], tuple(NNd[1:])
        dtype, dev = Mi.dtype, Mi.device
        B = Beff.to(dtype=dtype).reshape(N, -1, nT, 3)
        B = _ops._inner_contig(B, 2)
        M = _ops._inner_contig(Mi.reshape(N, -1, 3), 1)
        T1f, T2f, gf = (_flat_param(x, N, Nd, dev) for x in (T1, T2, γ))
        dtf = _ops.on_device(dt, dev).reshape(-1)
        K = _ops.beff_ckpt_interval(_ops.pick_ckpt_interval(dtf, T1f, T2f))
        flags = _ops.default_flags()
        Mo, ckpt = _ops.blochsim_beff_fwd(M, B, T1f, T2f, gf, dtf, K, flags)
        ctx.K, ctx.flags, ctx.relax = K, flags, T1 is not None
        saved = (Mo, ckpt, B, gf, dtf) + ((T1f, T2f) if T1 is not None else ())
        ctx.save_for_backward(*saved)
        ctx.NNd = NNd
        # a private copy is what backward reconstructs the states from: the caller may edit the returned tensor in place
        # (upstream returns a clone too, sims.py:128)
        return Mo.clone().reshape(NNd + (3,))

    @staticmethod
    def backward(ctx, grad_Mo: Tensor) -> Tuple[Optional[Tensor], Optional[Tensor], None, None, None, None]:
        r"""``grad_Mo`` `(N,*Nd,xyz)` -> ``grad_Mi`` `(N,*Nd,xyz)`, ``grad_Beff`` `(N,*Nd,nT,xyz)`, None*4."""
        need = ctx.needs_input_grad
        if not any(need[0:2]):                       # sims.py:153-157
            return None, None, None, None, None, None
        Mo, ckpt, B, gf, dtf, *rel = ctx.saved_tensors
        T1f, T2f = rel if ctx.relax else (None, None)
        N = B.shape[0]
        g = grad_Mo.to(dtype=Mo.dtype).reshape(N, -1, 3)
        g = _ops._inner_contig(g, 1)
        flags = ctx.flags | (_cabi.FLAG_NEED_GMI if need[0] else 0) | (_cabi.FLAG_NEED_GBEFF if need[1] else 0)
        gMi, gB = _ops.blochsim_beff_bwd(g, Mo, ckpt, B, T1f, T2f, gf, dtf, ctx.K, flags)
        grad_Mi = gMi.reshape(ctx.NNd + (3,)) if need[0] else None
        grad_Beff = gB.reshape(ctx.NNd + B.shape[-2:]) if need[1] else None
        return grad_Mi, grad_Beff, None, None, None, None


def blochsim(
    Mi: Tensor, Beff: Tensor, *,
    T1: Optional[Tensor] = None, T2: Optional[Tensor] = None,
    γ: Tensor = γH, dt: Tensor = dt0
) -> Tensor:
    r"""Bloch simulator with explicit Jacobian operation (differentiable w.r.t. ``Mi`` and ``Beff``).

    Usage:
        ``Mo = blochsim(Mi, Beff, *, T1, T2, γ, dt)``;  ``T1=T2=None`` ignores relaxation.
    Inputs:
        - ``Mi``: `(N, *Nd, xyz)`;  ``Beff``: `(N, *Nd, nT, xyz)`, "Gauss".
    Optionals:
        - ``T1``, ``T2``: `()` ⊻ `(N ⊻ 1, *Nd ⊻ 1,)` "Sec";  ``γ``: same, "Hz/Gauss";  ``dt``: `()` ⊻ `(N ⊻ 1,)` "Sec".
    Outputs:
        - ``Mo``: `(N, *Nd, xyz)`.
    There is no ``readout`` here: the receive signal summed inside the kernels comes from the fused path
    (``SpinArray.applypulse(pulse, readout=s)``).
    """
    assert (Mi.shape[:-1] == Beff.shape[:-2])        # sims.py:305
    Beff, ndim = Beff.to(Mi.device), Beff.ndim
    # host-resident constants (the defaults γH, dt0) first become their cached device copies, THEN views: the views'
    # base is then the same object on every call and the checkpoint-interval cache (no host sync) can hit
    γ, dt, T1, T2 = (_ops.on_device(x, Mi.device) for x in (γ, dt, T1, T2))
    γ, dt = (x.reshape(x.shape + (ndim - x.ndim) * (1,)) for x in (γ, dt))
    assert ((T1 is None) == (T2 is None))            # sims.py:311
    if T1 is not None:
        T1, T2 = (x.reshape(x.shape + (ndim - x.ndim) * (1,)) for x in (T1, T2))
    if Mi.dtype == torch.float32 and _ops.trig_policy() == 'strict':     # fp32 in and out, fp64 arithmetic
        return BlochSim.apply(Mi.double(), Beff.double(), T1, T2, γ, dt).float()
    return BlochSim.apply(Mi, Beff, T1, T2, γ, dt)


class FreePrec(Function):
    r"""Free precession with explicit Jacobian (differentiable w.r.t. ``Mi`` only; sims.py:318-421).

    One elementwise CUDA kernel (``mrphy_freeprec``); the backward applies the transposed map with the same kernel.
    """

    @staticmethod
    def forward(ctx, Mi: Tensor, dur: Tensor, T1: Optional[Tensor], T2: Optional[Tensor],
                Δf: Optional[Tensor]) -> Tensor:
        assert (T1 is None) == (T2 is None)
        _ops._require_cuda(Mi)
        N, Nd, dev = Mi.shape[0], tuple(Mi.shape[1:-1]), Mi.device
        args = (_ops.on_device(dur, dev).reshape(-1), _flat_param(T1, N, Nd, dev), _flat_param(T2, N, Nd, dev),
                _flat_param(Δf, N, Nd, dev))
        ctx.has = [x is not None for x in args]
        ctx.save_for_backward(*[x for x in args if x is not None])     # version-checked, unlike attributes on ctx
        ctx.shape = Mi.shape
        M = _ops._inner_contig(Mi.reshape(N, -1, 3), 1)
        return _ops.freeprec_cuda(M, *args, False).reshape(Mi.shape)

    @staticmethod
    def backward(ctx, grad_Mo: Tensor):
        if not ctx.needs_input_grad[0]:
            return None, None, None, None, None
        saved = list(ctx.saved_tensors)
        args = [saved.pop(0) if h else None for h in ctx.has]
        g = _ops._inner_contig(grad_Mo.reshape(ctx.shape[0], -1, 3), 1)
        return _ops.freeprec_cuda(g, *args, True).reshape(ctx.shape), None, None, None, None


def freeprec(
    Mi: Tensor, dur: Tensor, *,
    T1: Optional[Tensor] = None, T2: Optional[Tensor] = None,
    Δf: Optional[Tensor] = None
) -> Tensor:
    r"""Isochromats free precession with given relaxation and off-resonance (sims.py:424-458).

    - ``Mi``: `(N, *Nd, xyz)`;  ``dur``: `()` ⊻ `(N ⊻ 1,)` "Sec"
    - ``T1``, ``T2``: `()` ⊻ `(N ⊻ 1, *Nd ⊻ 1,)` "Sec";  ``Δf``: `(N ⊻ 1, *Nd ⊻ 1,)` "Hz"
    """
    ndim = Mi.ndim
    dur = dur.reshape(dur.shape + (ndim - dur.ndim) * (1,))
    assert ((T1 is None) == (T2 is None))
    if T1 is not None:
        T1, T2 = (x.reshape(x.shape + (ndim - x.ndim) * (1,)) for x in (T1, T2))
    if Δf is not None:
        Δf = Δf.reshape(Δf.shape + (ndim - 1 - Δf.ndim) * (1,))
    return FreePrec.apply(Mi, dur, T1, T2, Δf)
