r"""Pulse and spin containers of the ``mrphy`` API: ``Pulse``, ``SpinArray``, ``SpinCube``, ``Examples``.

Behavioural mirror of ``/root/reference/mrphy/mobjs.py`` -- same constructor keywords (Greek ones included),
same coercion of everything assigned to the object's device/dtype, same compact ``_`` storage with mask
embed/extract, same ``asdict`` keys and ``interpT`` grid -- written from scratch around a small
"normaliser per attribute" table.  ``SpinArray.applypulse`` is the entry of the hot path: it launches the fused
CUDA operator (``_ops.fused_applypulse``) instead of materialising ``Beff`` and stepping through time in Python
(mobjs.py:435-446 upstream).
"""
import copy
from typing import Optional

import numpy as np
import torch
from torch import Tensor, tensor

from mrphy import T1G, T2G, dt0, gmax0, rfmax0, smax0, γH, π
from mrphy import _ops, beffective, sims, utils

__all__ = ['Pulse', 'SpinArray', 'SpinCube', 'Examples']

OptT = Optional[Tensor]
_CPU = torch.device('cpu')
_F32 = torch.float32

# package defaults are fp64 CPU scalars; objects on a GPU get device-side clones of ONE cached copy instead of a
# synchronising host->device transfer per attribute and per object
_DEFAULTS = {id(c): c for c in (γH, dt0, gmax0, smax0, rfmax0, T1G, T2G)}
_on_device = {}


def _cast(value, device, dtype) -> Tensor:
    """Anything assignable -> tensor on (device, dtype)."""
    if not isinstance(value, Tensor):
        if isinstance(value, (int, float)) and device.type == 'cuda':
            return torch.full((), value, device=device, dtype=dtype)     # a fill kernel: no (synchronous) host->device copy
        return tensor(value, device=device, dtype=dtype)
    if device.type == 'cuda' and id(value) in _DEFAULTS:
        key = (id(value), device, dtype)
        if key not in _on_device:
            _on_device[key] = value.to(device=device, dtype=dtype)
        return _on_device[key].clone()
    return value.to(device=device, dtype=dtype)


def _detacher(to_numpy: bool):
    return (lambda t: t.detach().cpu().numpy()) if to_numpy else (lambda t: t.detach())


def _one_of(full, compact, extract):
    """The `x ⊻ x_` convention: at most one given; the non-compact form is extracted with the mask."""
    assert (full is None) or (compact is None)
    return compact if full is None else extract(full)


def _explicit_route(pulse, b1Map_, spin_inputs) -> bool:
    """Gradients w.r.t. spin inputs through the dense field and the explicit-``Beff`` kernels: only for more than 16
    transmit coils with a ``b1Map``, which the fused kernels do not take (everything else runs fused)."""
    many_coils = b1Map_ is not None and pulse.rf.ndim == 4 and pulse.rf.shape[3] > 16
    return many_coils and torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in spin_inputs)



def _mask_kernel_ok(v: Tensor) -> bool:
    """embed/extract run the one-pass CUDA gather for floating CUDA tensors; anything else (CPU objects, integer or
    boolean payloads) takes the equivalent torch indexing."""
    return v.is_cuda and v.dtype in (torch.float32, torch.float64) and v.numel() > 0 and v.ndim >= 2


class _Obj(object):
    """Attribute writes go through ``_store`` (validation + normalisation); deepcopy copies slots verbatim."""
    __slots__ = ()

    def __deepcopy__(self, memo):
        twin = object.__new__(type(self))
        memo[id(self)] = twin
        for klass in type(self).__mro__:
            for name in getattr(klass, '__slots__', ()):
                try:
                    object.__setattr__(twin, name, copy.deepcopy(object.__getattribute__(self, name), memo))
                except AttributeError:      # slot never filled (e.g. SpinArray slots of a SpinCube)
                    pass
        return twin

    def _put(self, **items):
        for name, value in items.items():
            object.__setattr__(self, name, value)


# ======================================================================================================
class Pulse(_Obj):
    r"""RF + gradient waveforms.

    ``Pulse(rf, gr, *, dt, gmax, smax, rfmax, desc, device, dtype)`` -- give ``rf`` `(N,xy,nT,(nCoils))` [Gauss]
    and/or ``gr`` `(N,xyz,nT)` [Gauss/cm]; a missing one is zero.  ``dt`` `()`⊻`(N⊻1,)` [s]; limits ``gmax``,
    ``smax`` `()`⊻`(N⊻1, xyz⊻1)`, ``rfmax`` `()`⊻`(N⊻1,(nCoils))`.

    Stored forms: ``dt`` `(N⊻1,)`, ``gmax``/``smax`` `(N⊻1, xyz)`, ``rfmax`` `(N⊻1,(nCoils))`; ``shape`` is
    `(N,1,nT)`.  ``device``, ``dtype``, ``is_cuda``, ``shape`` cannot be reassigned; everything else is moved to
    the pulse's device/dtype when set.
    """

    _readonly = ('device', 'dtype', 'is_cuda', 'shape')
    _limits = ('gmax', 'smax', 'rfmax')
    __slots__ = {'rf', 'gr', 'dt', 'desc', 'gmax', 'smax', 'rfmax', 'device', 'dtype', 'is_cuda', 'shape'}

    def __init__(
        self,
        rf: OptT = None,
        gr: OptT = None,
        *,
        dt: Tensor = dt0,
        gmax: Tensor = gmax0,
        smax: Tensor = smax0,
        rfmax: Tensor = rfmax0,
        desc: str = "generic pulse",
        device: torch.device = _CPU,
        dtype: torch.dtype = _F32,
    ):
        assert isinstance(device, torch.device) and isinstance(dtype, torch.dtype)
        assert rf is not None or gr is not None, "Missing both `rf` and `gr` inputs"
        given = rf if rf is not None else gr
        N, nT = given.shape[0], given.shape[2]
        self._put(device=device, dtype=dtype, is_cuda=(device.type == 'cuda'), shape=torch.Size((N, 1, nT)))
        zeros = lambda rows: torch.zeros((N, rows, nT), device=device, dtype=dtype)
        self.gr = zeros(3) if gr is None else gr
        self.rf = zeros(2) if rf is None else rf
        for name, value in (('dt', dt), ('gmax', gmax), ('smax', smax), ('rfmax', rfmax), ('desc', desc)):
            setattr(self, name, value)

    def __setattr__(self, name, value):
        if name in self._readonly:
            raise AttributeError(f"'Pulse' object attribute '{name}' is read-only")
        if name == 'desc':
            return object.__setattr__(self, name, value)
        t = _cast(value, self.device, self.dtype)
        if name in ('rf', 'gr'):
            assert t.shape[0] == self.shape[0] and t.shape[2] == self.shape[2]
        elif name == 'dt':
            t = t.reshape(1) if t.ndim == 0 else t
            assert t.ndim == 1
            if t.is_cuda and (not isinstance(value, Tensor) or (value.device.type == 'cpu' and not value.requires_grad)):
                # the value is known here without a device->host read: the checkpoint policy wants max(dt) on the host
                # (a Python float enters as float64, not torch's default float32, before it is rounded to the pulse's dtype)
                host = value if isinstance(value, Tensor) else torch.as_tensor(value, dtype=torch.float64)
                _ops.note_host_max(t, float(host.to(self.dtype).max()))
        elif name == 'rfmax':
            if t.ndim == 0:
                t = t.reshape(1)
            elif t.ndim == 2 and t.shape[1] == 1:
                t = t.squeeze(1)
        elif name in ('gmax', 'smax'):
            rows = 1 if t.ndim == 0 else t.shape[0]
            t = t.expand((rows, self.gr.shape[1]))
        object.__setattr__(self, name, t)

    # ---- conversions
    def asdict(self, *, toNumpy: bool = True) -> dict:
        r"""Detached data + ``desc, device, dtype``; ``Pulse(**pulse.asdict(toNumpy=False))`` rebuilds the pulse."""
        get = _detacher(toNumpy)
        out = {name: get(getattr(self, name)) for name in ('rf', 'gr', 'dt') + self._limits}
        for name in ('desc', 'device', 'dtype'):
            out[name] = getattr(self, name)
        return out

    def to(self, *, device: torch.device = _CPU, dtype: torch.dtype = _F32) -> 'Pulse':
        r"""This pulse on another device/dtype (``self`` if nothing changes; limits reset to defaults as upstream)."""
        unchanged = (self.device, self.dtype) == (device, dtype)
        return self if unchanged else Pulse(self.rf, self.gr, dt=self.dt, desc=self.desc, device=device, dtype=dtype)

    # ---- physics
    def beff(self, loc: Tensor, *, Δf: OptT = None, b1Map: OptT = None, γ: Tensor = γH) -> Tensor:
        r"""B-effective `(N,*Nd,nT,xyz)` [Gauss] seen at ``loc`` `(N,*Nd,xyz)` [cm]; optional ``Δf`` `(N,*Nd)` [Hz],
        ``b1Map`` `(N,*Nd,xy,(nCoils))`, ``γ`` [Hz/Gauss]."""
        here = lambda t: None if t is None else t.to(device=self.device)
        return beffective.rfgr2beff(self.rf, self.gr, here(loc), Δf=here(Δf), b1Map=here(b1Map), γ=here(γ))

    def interpT(self, dt: Tensor, *, kind: str = 'linear', differentiable: bool = False) -> 'Pulse':
        r"""Resample to the (single, global) dwell time ``dt``; ``kind`` as in ``scipy.interpolate.interp1d``.

        Samples sit at the END of their interval and a zero sample is implied at t=0.  The new length is
        ``t_end // dt_new`` in Python floats, exactly as upstream (mobjs.py:211-212): nT=10 at 4 µs -> 2 µs gives
        19 samples.  ``kind='linear'`` is evaluated on the pulse's device with NO device->host read: the dwell times are
        taken from the host values the tensors were made from (a CUDA ``dt`` of unknown origin costs one read, cached per
        tensor), so a multi-scale design loop stays free of host synchronisation.  Other kinds take the scipy host round
        trip like upstream.  By default the result carries no autograd history (as upstream); with
        ``differentiable=True`` (linear kind) gradients flow from the resampled ``rf``/``gr`` back to this pulse's.
        The result has default limits.
        """
        assert self.dt.numel() == 1 and dt.numel() == 1
        host = lambda t: _ops._cached_max(t) if t.is_cuda else float(t.reshape(-1)[0])
        old, new = host(self.dt), host(dt)
        if old == new:
            return copy.deepcopy(self)
        nT = self.shape[2]
        kw = {'device': self.device, 'dtype': self.dtype}
        n_new = int((nT * old) // new)                 # == len(np.arange(1, t_end // dt_new + 1)), mobjs.py:211-212
        if kind == 'linear':
            # knots k*old and query points j*new, their bracketing and weights: the same IEEE double operations as upstream's
            # numpy grid, evaluated on the pulse's device (nothing is uploaded, nothing is read back)
            f8 = {'device': self.device, 'dtype': torch.float64}
            knots_t = torch.arange(0, nT + 1, **f8) * old
            query_t = torch.arange(1, n_new + 1, **f8) * new
            right_t = torch.searchsorted(knots_t, query_t).clamp_(1, nT)
            lo_t, hi_t = knots_t.index_select(0, right_t - 1), knots_t.index_select(0, right_t)
            frac_t = (query_t - lo_t) / (hi_t - lo_t)

            def resample(x):
                x = x if differentiable else x.detach()
                padded = torch.cat((torch.zeros_like(x[:, :, :1]), x), dim=2).double()
                w = frac_t.reshape((1, 1, -1) + (1,) * (x.ndim - 3))
                lo, hi = padded.index_select(2, right_t - 1), padded.index_select(2, right_t)
                return (lo + (hi - lo) * w).to(**kw)
        else:
            assert not differentiable, 'only the linear kind is differentiable'
            from scipy import interpolate
            knots = np.arange(0, nT + 1) * old
            query = np.arange(1, knots[-1] // new + 1) * new

            def resample(x):
                padded = torch.cat((torch.zeros_like(x[:, :, :1]), x.detach()), dim=2).cpu().numpy()
                f = interpolate.interp1d(knots, padded, axis=2, kind=kind, copy=False, assume_sorted=True)
                return tensor(f(query), **kw)

        # dt goes in as the host value: the new pulse's dwell time is then known without a device read as well
        return Pulse(resample(self.rf), resample(self.gr), dt=new,
                     desc=f"{self.desc} + interpT\'ed: dt = {new}", **kw)


# ======================================================================================================
class SpinArray(_Obj):
    r"""Spins on a masked regular array.

    ``SpinArray(shape, mask, *, T1⊻T1_, T2⊻T2_, γ⊻γ_, M⊻M_, device, dtype)`` with ``shape`` = `(N, *Nd)` and a
    boolean ``mask`` `(1, *Nd)` shared by the batch (default: all true).  Only the ``nM`` masked spins are stored,
    in the *compact* attributes ``T1_``, ``T2_``, ``γ_`` `(N, nM)` and ``M_`` `(N, nM, xyz)`; reading ``T1``,
    ``T2``, ``γ``, ``M`` embeds them into `(N, *Nd, ...)` (NaN outside the mask), assigning extracts.  Defaults:
    grey-matter T1/T2, proton γ, M = [0,0,1].  Do not modify ``mask``; in-place edits of an embedded view do not
    reach the compact data -- index the compact arrays through :meth:`crds_` instead.
    """

    _readonly = ('shape', 'mask', 'device', 'dtype', 'is_cuda', 'ndim', 'nM', 'midx', 'minv')
    _compact = ('T1_', 'T2_', 'γ_', 'M_')
    __slots__ = {'T1_', 'T2_', 'γ_', 'M_', 'shape', 'mask', 'ndim', 'nM', 'device', 'dtype', 'is_cuda', 'midx', 'minv'}

    def __init__(
        self,
        shape: tuple,
        mask: OptT = None,
        *,
        T1: OptT = None,
        T1_: OptT = None,
        T2: OptT = None,
        T2_: OptT = None,
        γ: OptT = None,
        γ_: OptT = None,
        M: OptT = None,
        M_: OptT = None,
        device: torch.device = _CPU,
        dtype: torch.dtype = _F32,
    ):
        shape = tuple(shape)
        if mask is None:
            mask = torch.ones((1,) + shape[1:], dtype=torch.bool, device=device)
        mask = mask.to(device=device)
        assert isinstance(device, torch.device) and isinstance(dtype, torch.dtype)
        assert mask.dtype == torch.bool and mask.shape == (1,) + shape[1:]
        # flat positions of the stored spins, found once: embed/extract are then an index_copy_/index_select on the
        # device with no host synchronisation (boolean-mask indexing would run nonzero() + a sync on every call)
        midx = mask.reshape(-1).nonzero().reshape(-1)
        # inverse map (-1 outside the mask): embed is then ONE gather pass with the NaN padding fused (mask_copy kernel)
        minv = torch.full((mask.numel(),), -1, dtype=torch.int64, device=device)
        minv[midx] = torch.arange(midx.numel(), dtype=torch.int64, device=device)
        self._put(shape=shape, mask=mask, ndim=len(shape), nM=int(midx.numel()), device=device,
                  dtype=dtype, is_cuda=(device.type == 'cuda'), midx=midx, minv=minv)
        fallback = {'T1': T1G, 'T2': T2G, 'γ': γH, 'M': tensor([0., 0., 1.])}
        for name, full, compact in (('T1', T1, T1_), ('T2', T2, T2_), ('γ', γ, γ_), ('M', M, M_)):
            assert (full is None) or (compact is None)
            if full is not None:
                setattr(self, name, full)
            else:
                setattr(self, name + '_', fallback[name] if compact is None else compact)

    def _covers_grid(self) -> bool:
        return self.nM == int(np.prod(self.shape[1:]))

    def __getattr__(self, name):     # reached only for names without a slot value: the embedded views
        if name + '_' not in self._compact:
            raise AttributeError(f"'SpinArray' has no attribute '{name}'")
        stored = getattr(self, name + '_')
        return stored.reshape(self.shape + stored.shape[2:]) if self._covers_grid() else self.embed(stored)

    def __setattr__(self, name, value):
        if name in self._readonly:
            raise AttributeError(f"'SpinArray' object attribute '{name}' is read-only")
        t = _cast(value, self.device, self.dtype)
        N = self.shape[0]
        if name + '_' in self._compact:          # embedded form given: broadcast over the grid, keep masked spins
            name += '_'
            t = self.extract(t.expand(self.shape + ((3,) if name == 'M_' else ())))
        if name == 'M_':
            if t.shape != (N, self.nM, 3):
                t = t.expand((N, self.nM, 3)).clone()
        elif name in self._compact:
            t = t.expand((N, self.nM))           # stride-0 when a scalar was given
        object.__setattr__(self, name, t)

    # ---- mask plumbing
    def embed(self, v_: Tensor, *, out: OptT = None) -> Tensor:
        r"""Compact `(N,nM,...)` -> `(N,*Nd,...)`; positions outside the mask are NaN (or keep ``out``'s content)."""
        if out is None and _mask_kernel_ok(v_):
            flat = _ops.mask_copy_cuda(v_.reshape(v_.shape[0], v_.shape[1], -1).contiguous(), self.minv, self.midx, False)
            return flat.reshape((v_.shape[0],) + self.shape[1:] + v_.shape[2:])
        if out is None:
            out = v_.new_full(self.shape + v_.shape[2:], float('nan'))
        if out.is_contiguous():
            out.view((self.shape[0], -1) + v_.shape[2:]).index_copy_(1, self.midx, v_.to(out.dtype))
        else:
            out[self.mask.expand(self.shape)] = v_.reshape((-1,) + v_.shape[2:])
        return out

    def extract(self, v: Tensor, *, out_: OptT = None) -> Tensor:
        r"""`(N,*Nd,...)` -> compact `(N,nM,...)`, row-major over `*Nd`."""
        tail = v.shape[self.ndim:]
        if _mask_kernel_ok(v):
            chosen = _ops.mask_copy_cuda(v.reshape(v.shape[0], self.minv.numel(), -1).contiguous(), self.midx, self.minv, False)
            chosen = chosen.reshape((v.shape[0], self.nM) + tail)
        else:
            chosen = v.reshape((v.shape[0], -1) + tail).index_select(1, self.midx)
        if out_ is None:
            return chosen
        out_.copy_(chosen)
        return out_

    def crds_(self, crds: list) -> list:
        r"""Translate an index list for `(N,*Nd,...)` arrays into one for the compact `(N,nM,...)` arrays:
        ``v_[spinarray.crds_(crds)]`` addresses ``v[crds]``, and assignments through it reach the stored data."""
        assert len(crds) >= self.ndim
        lookup = torch.full(self.mask.shape, -1, dtype=torch.int64)
        lookup[self.mask.cpu()] = torch.arange(self.nM)
        hits = lookup[tuple([[0]] + list(crds[1:self.ndim]))].tolist()
        return [crds[0], [h for h in hits if h != -1]] + list(crds[self.ndim:])

    def mask_(self, *, mask: Tensor) -> Tensor:
        r"""Restrict an external ``mask`` `(1,*Nd)` to the stored spins -> `(1,nM)`.  (Upstream's version calls a
        tensor and always raises, mobjs.py:605.)"""
        return mask.to(self.device).reshape(1, -1).index_select(1, self.midx)

    def dim(self) -> int:
        r"""Number of dimensions of ``shape``."""
        return len(self.shape)

    def numel(self) -> int:
        r"""Grid points including masked-out ones."""
        return self.mask.numel()

    def size(self) -> tuple:
        r"""Alias of ``shape``."""
        return self.shape

    # ---- conversions
    def asdict(self, *, toNumpy: bool = True, doEmbed: bool = True) -> dict:
        r"""Detached ``T1, T2, γ, M`` (embedded, or the ``_`` forms with ``doEmbed=False``), ``mask``, ``shape``,
        ``device``, ``dtype``."""
        get = _detacher(toNumpy)
        out = {name: get(getattr(self, name)) for name in (('T1', 'T2', 'γ', 'M') if doEmbed else self._compact)}
        out['mask'] = get(self.mask)
        for name in ('shape', 'device', 'dtype'):
            out[name] = getattr(self, name)
        return out

    def to(self, *, device: torch.device = _CPU, dtype: torch.dtype = _F32) -> 'SpinArray':
        r"""This spin array on another device/dtype (``self`` if nothing changes)."""
        if (self.device, self.dtype) == (device, dtype):
            return self
        return SpinArray(self.shape, self.mask, T1_=self.T1_, T2_=self.T2_, γ_=self.γ_, M_=self.M_, device=device,
                         dtype=dtype)

    # ---- physics
    def applypulse(
        self,
        pulse: Pulse,
        *,
        loc: OptT = None,
        loc_: OptT = None,
        Δf: OptT = None,
        Δf_: OptT = None,
        b1Map: OptT = None,
        b1Map_: OptT = None,
        doEmbed: bool = False,
        doRelax: bool = True,
        doUpdate: bool = False,
        record: Optional[int] = None,
    ):
        r"""Simulate ``pulse`` on these spins and return the magnetisation.

        ``loc`` ⊻ ``loc_`` `(N,*Nd ⊻ nM,xyz)` [cm] is required; ``Δf`` ⊻ ``Δf_`` `(N,*Nd ⊻ nM)` [Hz] and ``b1Map`` ⊻
        ``b1Map_`` `(N,*Nd ⊻ nM,xy,(nCoils))` are optional.  ``doRelax=False`` ignores T1/T2; ``doUpdate`` stores
        the result in ``M_`` (with its autograd graph, as upstream); ``doEmbed`` returns `(N,*Nd,xyz)` instead of
        the compact `(N,nM,xyz)`.

        All ``nT`` steps run in one fused CUDA kernel and gradients reach ``pulse.rf``, ``pulse.gr`` and ``M_``, and
        ``loc``/``Δf``/``b1Map``/``γ`` when they require grad (upstream's autograd through rfgr2beff; the fused backward
        forms these per-spin sums without materialising the field).  Only more than 16 transmit coils with a ``b1Map``,
        which the fused kernels do not take, materialise the field (``pulse2beff``) and run the explicit-``Beff``
        kernels, whose per-spin pass takes at most 16 coils as well.

        ``record = s`` (an integer, 1 <= s <= nT) also returns the magnetisation during the pulse: ``(M, Mt)``, ``Mt``
        `(N,nM,nR,xyz)` (`(N,*Nd,nR,xyz)` with ``doEmbed``), nR = nT // s, ``Mt[..., r, :]`` the state after (r+1)·s
        steps -- ``M`` of the pulse cut to its first (r+1)·s samples.  Compact ``Mt`` is a non-contiguous view.
        ``doUpdate`` stores ``M`` only.  Gradients flow through both.  Refused (ValueError) beyond 16 transmit coils
        with a ``b1Map``: the explicit-``Beff`` route does not record.
        """
        assert (loc_ is None) != (loc is None)
        loc_ = loc_ if loc is None else self.extract(loc)
        Δf_ = _one_of(Δf, Δf_, self.extract)
        b1Map_ = _one_of(b1Map, b1Map_, self.extract)
        T1_, T2_ = (self.T1_, self.T2_) if doRelax else (None, None)
        if record is not None:
            p = pulse.to(device=self.device, dtype=self.dtype)
            M_, Mt_ = _ops.fused_applypulse(self.M_, p.rf, p.gr, loc_, Δf_=Δf_, b1Map_=b1Map_, T1_=T1_, T2_=T2_,
                                            γ_=self.γ_, dt=p.dt, record=record)
            if doUpdate:
                self.M_ = M_
            return (self.embed(M_), self.embed(Mt_)) if doEmbed else (M_, Mt_)
        if _explicit_route(pulse, b1Map_, (loc_, Δf_, b1Map_, self.γ_)):
            beff_ = self.pulse2beff(pulse, loc_=loc_, Δf_=Δf_, b1Map_=b1Map_)
            M_ = sims.blochsim(self.M_, beff_, T1=T1_, T2=T2_, γ=self.γ_, dt=pulse.dt)
        else:
            p = pulse.to(device=self.device, dtype=self.dtype)
            M_ = _ops.fused_applypulse(self.M_, p.rf, p.gr, loc_, Δf_=Δf_, b1Map_=b1Map_, T1_=T1_, T2_=T2_,
                                       γ_=self.γ_, dt=p.dt)
        if doUpdate:
            self.M_ = M_
        return self.embed(M_) if doEmbed else M_

    def freeprec(
        self,
        dur: Tensor,
        *,
        Δf: OptT = None,
        Δf_: OptT = None,
        doEmbed: bool = False,
        doRelax: bool = True,
        doUpdate: bool = False,
    ) -> Tensor:
        r"""Free precession for ``dur`` `()`⊻`(N⊻1,)` [s] with optional off-resonance ``Δf`` ⊻ ``Δf_``; flags as in
        :meth:`applypulse`."""
        Δf_ = _one_of(Δf, Δf_, self.extract)
        T1_, T2_ = (self.T1_, self.T2_) if doRelax else (None, None)
        M_ = sims.freeprec(self.M_, dur.to(self.device), T1=T1_, T2=T2_, Δf=Δf_)
        if doUpdate:
            self.M_ = M_
        return self.embed(M_) if doEmbed else M_

    def applysequence(
        self,
        events,
        *,
        loc: OptT = None,
        loc_: OptT = None,
        Δf: OptT = None,
        Δf_: OptT = None,
        b1Map: OptT = None,
        b1Map_: OptT = None,
        doEmbed: bool = False,
        doRelax: bool = True,
        doUpdate: bool = False,
    ) -> Tensor:
        r"""A whole sequence -- pulses and free-precession gaps in order -- without returning to the objects between stages.

        ``events`` is an iterable of :class:`Pulse` (simulated like :meth:`applypulse`) and durations (``Tensor`` `()`⊻`(N⊻1,)`
        or float, seconds; free precession like :meth:`freeprec`).  Equivalent to chaining the two methods with
        ``doUpdate=True`` (mobjs.py:394-450, 555-592), but the magnetisation stays a compact device tensor from the first
        kernel to the last -- no embed / extract / attribute coercion per stage, no host synchronisation -- and the result is
        differentiable w.r.t. every pulse's ``rf`` / ``gr``, ``M_`` and the spin inputs as in :meth:`applypulse`.  The chain is CUDA-graph capturable as a whole
        (``mrphy.graphs.capture``): one replay per sequence.  Arguments and flags as in :meth:`applypulse`.
        """
        assert (loc_ is None) != (loc is None)
        loc_ = loc_ if loc is None else self.extract(loc)
        Δf_ = _one_of(Δf, Δf_, self.extract)
        b1Map_ = _one_of(b1Map, b1Map_, self.extract)
        T1_, T2_ = (self.T1_, self.T2_) if doRelax else (None, None)
        M_ = self.M_
        for ev in events:
            if isinstance(ev, Pulse):
                p = ev.to(device=self.device, dtype=self.dtype)
                if _explicit_route(p, b1Map_, (loc_, Δf_, b1Map_, self.γ_)):
                    beff_ = p.beff(loc_, γ=self.γ_, Δf=Δf_, b1Map=b1Map_)
                    M_ = sims.blochsim(M_, beff_, T1=T1_, T2=T2_, γ=self.γ_, dt=p.dt)
                else:
                    M_ = _ops.fused_applypulse(M_, p.rf, p.gr, loc_, Δf_=Δf_, b1Map_=b1Map_, T1_=T1_, T2_=T2_, γ_=self.γ_,
                                               dt=p.dt)
            else:
                dur = ev if isinstance(ev, Tensor) else tensor(float(ev), dtype=torch.float64)
                M_ = sims.freeprec(M_, _ops.on_device(dur, self.device), T1=T1_, T2=T2_, Δf=Δf_)
        if doUpdate:
            self.M_ = M_
        return self.embed(M_) if doEmbed else M_

    def pulse2beff(
        self,
        pulse: Pulse,
        *,
        loc: OptT = None,
        loc_: OptT = None,
        Δf: OptT = None,
        Δf_: OptT = None,
        b1Map: OptT = None,
        b1Map_: OptT = None,
        doEmbed: bool = False,
    ) -> Tensor:
        r"""B-effective `(N,*Nd ⊻ nM,nT,xyz)` of ``pulse`` at these spins (their ``γ``); arguments as in
        :meth:`applypulse`."""
        assert (loc_ is None) != (loc is None)
        loc_ = loc_ if loc is None else self.extract(loc)
        Δf_ = _one_of(Δf, Δf_, self.extract)
        b1Map_ = _one_of(b1Map, b1Map_, self.extract)
        p = pulse.to(device=self.device, dtype=self.dtype)
        beff_ = p.beff(loc_, γ=self.γ_, Δf=Δf_, b1Map=b1Map_)
        return self.embed(beff_) if doEmbed else beff_


# ======================================================================================================
class SpinCube(SpinArray):
    r"""A :class:`SpinArray` with regular-grid geometry.

    ``SpinCube(shape, fov, *, mask, ofst, Δf⊻Δf_, T1⊻T1_, T2⊻T2_, γ⊻γ_, M⊻M_, device, dtype)``; ``fov`` and
    ``ofst`` are `(N, xyz)` [cm].  Adds ``loc_`` `(N, nM, xyz)` [cm] (read-only, recomputed whenever ``fov`` or
    ``ofst`` is assigned: ``fov·(index − n//2)/n + ofst``), ``Δf_`` `(N, nM)` [Hz] and ``spinarray`` (the underlying
    :class:`SpinArray`, to which every other attribute is forwarded).
    """

    _readonly = ('spinarray', 'loc_')
    _compact = ('Δf_', 'loc_')
    __slots__ = {'spinarray', 'loc_', 'Δf_', 'fov', 'ofst'}

    def __init__(
        self,
        shape: tuple,
        fov: Tensor,
        *,
        mask: OptT = None,
        ofst: Tensor = tensor([[0., 0., 0.]]),
        Δf: OptT = None,
        Δf_: OptT = None,
        T1: OptT = None,
        T1_: OptT = None,
        T2: OptT = None,
        T2_: OptT = None,
        γ: OptT = None,
        γ_: OptT = None,
        M: OptT = None,
        M_: OptT = None,
        device: torch.device = _CPU,
        dtype: torch.dtype = _F32,
    ):
        core = SpinArray(shape, mask, T1=T1, T1_=T1_, T2=T2, T2_=T2_, γ=γ, γ_=γ_, M=M, M_=M_, device=device, dtype=dtype)
        kw = {'device': core.device, 'dtype': core.dtype}
        self._put(spinarray=core, fov=fov.to(**kw), ofst=ofst.to(**kw),
                  loc_=torch.zeros((core.shape[0], core.nM, 3), **kw))
        self._update_loc_()
        assert (Δf is None) or (Δf_ is None)
        if Δf is not None:
            self.Δf = Δf
        else:
            self.Δf_ = tensor(0.) if Δf_ is None else Δf_

    def __getattr__(self, name):
        core = object.__getattribute__(self, 'spinarray')    # never via self.<attr>: a half-built copy would recurse
        if name + '_' in self._compact:
            stored = getattr(self, name + '_')
            return stored.reshape(core.shape + stored.shape[2:]) if core._covers_grid() else core.embed(stored)
        try:
            return getattr(core, name)
        except AttributeError:
            raise AttributeError(f"'SpinCube' has no attribute '{name}'")

    def __setattr__(self, name, value):
        if name in self._readonly or name + '_' in self._readonly:
            raise AttributeError(f"'SpinCube' object attribute '{name}' is read-only")
        core = self.spinarray
        if name in SpinArray.__slots__ or name + '_' in SpinArray.__slots__:
            return setattr(core, name, value)
        t = _cast(value, core.device, core.dtype)
        if name + '_' in self._compact:
            name += '_'
            t = core.extract(t.expand(core.shape))
        if name == 'Δf_':
            t = t.expand((core.shape[0], core.nM))
        elif name in ('fov', 'ofst'):
            assert t.ndim == 2
        object.__setattr__(self, name, t)
        if name in ('fov', 'ofst'):
            self._update_loc_()

    def _update_loc_(self):
        r"""Refresh ``loc_`` in place from ``fov`` and ``ofst``; the grid is centred on index ``n//2``."""
        core = self.spinarray
        kw = {'device': core.device, 'dtype': core.dtype}
        ticks = [(torch.arange(n, **kw) - utils.ctrsub(n)) / n for n in core.shape[1:]]
        inside = core.mask[0]
        for axis, grid in enumerate(torch.meshgrid(*ticks, indexing='ij')):
            self.loc_[..., axis] = self.fov[:, None, axis] * grid[inside][None] + self.ofst[:, None, axis]

    # ---- conversions
    def asdict(self, *, toNumpy: bool = True, doEmbed: bool = True) -> dict:
        r"""``loc``, ``Δf``, ``fov``, ``ofst`` plus everything :meth:`SpinArray.asdict` returns."""
        get = _detacher(toNumpy)
        out = {'loc': get(self.loc), 'Δf': get(self.Δf), 'fov': self.fov, 'ofst': self.ofst}
        out.update(self.spinarray.asdict(toNumpy=toNumpy, doEmbed=doEmbed))
        return out

    def to(self, *, device: torch.device = _CPU, dtype: torch.dtype = _F32) -> 'SpinCube':
        r"""This cube on another device/dtype (``self`` if nothing changes)."""
        if (self.device, self.dtype) == (device, dtype):
            return self
        return SpinCube(self.shape, self.fov, mask=self.mask, ofst=self.ofst, Δf_=self.Δf_, T1_=self.T1_,
                        T2_=self.T2_, γ_=self.γ_, M_=self.M_, device=device, dtype=dtype)

    # ---- physics: the cube supplies its own geometry and off-resonance
    def applypulse(
        self,
        pulse: Pulse,
        *,
        b1Map: OptT = None,
        b1Map_: OptT = None,
        doEmbed: bool = False,
        doRelax: bool = True,
        doUpdate: bool = False,
        record: Optional[int] = None,
    ):
        r"""As :meth:`SpinArray.applypulse` with the cube's ``loc_`` and ``Δf_``; only ``b1Map`` ⊻ ``b1Map_`` is given."""
        b1Map_ = _one_of(b1Map, b1Map_, self.extract)
        return self.spinarray.applypulse(pulse, loc_=self.loc_, Δf_=self.Δf_, b1Map_=b1Map_, doEmbed=doEmbed,
                                         doRelax=doRelax, doUpdate=doUpdate, record=record)

    def applysequence(self, events, *, b1Map: OptT = None, b1Map_: OptT = None, doEmbed: bool = False, doRelax: bool = True,
                      doUpdate: bool = False) -> Tensor:
        r"""As :meth:`SpinArray.applysequence` with the cube's ``loc_`` and ``Δf_``."""
        b1Map_ = _one_of(b1Map, b1Map_, self.extract)
        return self.spinarray.applysequence(events, loc_=self.loc_, Δf_=self.Δf_, b1Map_=b1Map_, doEmbed=doEmbed,
                                            doRelax=doRelax, doUpdate=doUpdate)

    def freeprec(self, dur: Tensor, *, doEmbed: bool = False, doRelax: bool = True, doUpdate: bool = False) -> Tensor:
        r"""As :meth:`SpinArray.freeprec` with the cube's ``Δf_``."""
        return self.spinarray.freeprec(dur, Δf_=self.Δf_, doEmbed=doEmbed, doRelax=doRelax, doUpdate=doUpdate)

    def pulse2beff(self, pulse: Pulse, *, b1Map: OptT = None, b1Map_: OptT = None, doEmbed: bool = False) -> Tensor:
        r"""As :meth:`SpinArray.pulse2beff` with the cube's ``loc_`` and ``Δf_``.  (Upstream passes ``loc_``
        positionally to a keyword-only parameter and raises, mobjs.py:942.)"""
        return self.spinarray.pulse2beff(pulse, loc_=self.loc_, Δf_=self.Δf_, b1Map=b1Map, b1Map_=b1Map_,
                                         doEmbed=doEmbed)


class SpinBolus(SpinArray):
    """Placeholder kept for name compatibility (mobjs.py:968-973)."""

    def __init__(self):
        pass


# ======================================================================================================
class Examples(object):
    r"""Ready-made toy objects (mobjs.py:976-1038)."""

    @staticmethod
    def _cross_mask() -> Tensor:
        m = torch.zeros((1, 3, 3, 3), dtype=torch.bool)
        m[0, :, 1, :] = True
        m[0, 1, :, :] = True
        return m

    @staticmethod
    def pulse() -> Pulse:
        r"""512 samples: 10 G rf turning once around, unit x/y gradients, an arctan ramp on z."""
        nT = 512
        t = torch.arange(0, nT, dtype=_F32).reshape((1, 1, nT))
        turn = t / nT * 2 * π
        flat = torch.ones((1, 1, nT), dtype=_F32)
        rf = 10 * torch.cat([torch.cos(turn), torch.sin(turn)], 1)
        gr = torch.cat([flat, flat, 10 * torch.atan(t - round(nT / 2)) / π], 1)
        return Pulse(rf=rf, gr=gr, dt=dt0, device=_CPU, dtype=_F32)

    @staticmethod
    def spinarray() -> SpinArray:
        r"""15 spins on a 3×3×3 grid (a cross-shaped mask), T1 = 1 s, T2 = 40 ms."""
        return SpinArray((1, 3, 3, 3), mask=Examples._cross_mask(), T1_=tensor([[1.]]), T2_=tensor([[4e-2]]), γ_=γH,
                         device=_CPU, dtype=_F32)

    @staticmethod
    def spincube() -> SpinCube:
        r"""The same spins with a 3 cm field of view, a 1 cm z offset and Δf cancelling unit x/y gradients."""
        cube = SpinCube((1, 3, 3, 3), tensor([[3., 3., 3.]]), mask=Examples._cross_mask(), ofst=tensor([[0., 0., 1.]]),
                        T1_=tensor([[1.]]), T2_=tensor([[4e-2]]), γ_=γH, device=_CPU, dtype=_F32)
        cube.Δf = -cube.loc[0:1, :, :, :, 0:2].sum(dim=-1) * γH
        return cube
