"""torch.library custom ops over the C ABI (the only place tensors meet libmrphy_b200.so).

``mrphy_b200::blochsim_fused_fwd / _bwd`` implement, in one kernel each, what the reference does
with ``beffective.rfgr2beff`` (beffective.py:107-168) followed by ``sims.BlochSim.forward`` /
``.backward`` (sims.py:31-269) and the autograd of ``rfgr2beff``.  ``fused_applypulse`` is the
Python-level entry used by ``mobjs.SpinArray.applypulse`` (mobjs.py:394-450).
"""
import ctypes
import numbers
import os
import weakref
from typing import Optional, Tuple

import torch
from torch import Tensor

from mrphy import _cabi

_F = (torch.float32, torch.float64)
K_MAX = 64                  # checkpoint interval cap == staged chunk length (csrc: TCMAX)
K_MAX1 = 128                # ... of the fp32 single-coil kernels (csrc: MRPHY_TCMAX1)
TC_K_MAX = 32               # ... of the tensor-core multi-coil kernels (fp32, >= 3 coils with a b1Map; csrc: TC_TCMAX)
_AMPLIFY_BUDGET = 0.4       # resync before exp(K*dt/T2) exceeds e^0.4 ~ 1.5 (time-reversed states)


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError('mrphy (B200): the Bloch-simulation path is CUDA-only (sm_100a); got a '
                               f'{t.device} tensor. There is no CPU fallback.')


def _param(t: Optional[Tensor], N: int, nM: int, per_batch_only=False) -> _cabi.Param:
    """(N|1, nM|1) (or any shape broadcastable to it) -> pointer + element strides, no copy."""
    p = _cabi.Param()
    if t is None:
        return p
    if t.dtype not in _F:
        raise TypeError(f'mrphy (B200): float32/float64 expected, got {t.dtype}')
    v = t
    while v.ndim > 2 and v.shape[-1] == 1:   # (N,nM,1,1) style tails from sims.blochsim
        v = v[..., 0]
    if per_batch_only:
        v = v.reshape(-1)
        assert v.numel() in (1, N), 'dt must be () or (N|1,)'
        p.ptr, p.sn, p.sm = v.data_ptr(), (v.stride(0) if v.numel() == N and N > 1 else 0), 0
    else:
        while v.ndim < 2:
            v = v[None] if v.ndim == 0 else v[:, None]
        assert v.ndim == 2 and v.shape[0] in (1, N) and v.shape[1] in (1, nM), \
            f'per-spin constant of shape {tuple(t.shape)} does not broadcast to ({N},{nM})'
        p.ptr = v.data_ptr()
        p.sn = v.stride(0) if v.shape[0] == N and N > 1 else 0
        p.sm = v.stride(1) if v.shape[1] == nM and nM > 1 else 0
    p.f64 = int(v.dtype == torch.float64)
    return p


_const_cache = {}


def on_device(x: Optional[Tensor], device, dtype=None) -> Optional[Tensor]:
    """``x`` on ``device`` (and ``dtype`` when given).  Small host-resident constants -- the module defaults γH, dt0,
    T1G, T2G or a user's CPU scalars -- map to the SAME device tensor on every call (keyed by object and in-place version,
    weak references guard against id reuse): repeated calls neither pay a pageable host-to-device copy per constant
    nor defeat the per-tensor cache of `pick_ckpt_interval`.  The result is shared: callers never write to it."""
    if x is None:
        return None
    if x.device == device and (dtype is None or x.dtype == dtype):
        return x
    if x.device.type == 'cpu' and x.numel() <= 16 and not x.requires_grad:
        key = (id(x), device, dtype)
        hit = _const_cache.get(key)
        if hit is not None and hit[0]() is x and hit[1] == x._version:
            return hit[2]
        y = x.to(device=device) if dtype is None else x.to(device=device, dtype=dtype)
        if len(_const_cache) > 256:
            _const_cache.clear()
        _const_cache[key] = (weakref.ref(x), x._version, y)
        return y
    return x.to(device=device) if dtype is None else x.to(device=device, dtype=dtype)


def flat_param(x: Optional[Tensor], N: int, Nd: tuple, device) -> Optional[Tensor]:
    """(), (N|1,), (N|1, *Nd|1.., [1, 1])-style constant -> (N|1, nM|1) view (copy only for partial broadcasts)."""
    if x is None:
        return None
    x = on_device(x, device)
    while x.ndim > 1 + len(Nd):
        assert x.shape[-1] == 1
        x = x[..., 0]
    if x.ndim == 0:
        return x.reshape(1, 1)
    if all(s == 1 for s in x.shape[1:]):
        return x.reshape(x.shape[0], 1)
    x = x.reshape(x.shape + (1,) * (1 + len(Nd) - x.ndim))
    return x.expand((x.shape[0],) + tuple(Nd)).reshape(x.shape[0], -1)


def _inner_contig(t: Tensor, inner: int) -> Tensor:
    """Make the trailing `inner` dims densely packed (leading strides stay free)."""
    exp = 1
    for d in range(t.ndim - 1, t.ndim - 1 - inner, -1):
        if t.shape[d] != 1 and t.stride(d) != exp:
            return t.contiguous()
        exp *= t.shape[d]
    return t


def _bstride(t: Tensor, d: int) -> int:
    return t.stride(d) if t.shape[d] > 1 else 0


def _fill_common(a, Mi, rf, gr, loc, df, b1, T1, T2, gamma, dt, K, flags):
    N, nM = loc.shape[0], loc.shape[1]
    a.dtype = _cabi.MRPHY_F64 if loc.dtype == torch.float64 else _cabi.MRPHY_F32
    a.N, a.nM, a.nT = N, nM, rf.shape[2]
    a.nC = rf.shape[3] if rf.ndim == 4 else 1
    a.K = K
    a.flags = flags | (_cabi.FLAG_RF_COIL_DIM if rf.ndim == 4 else 0)
    if Mi is not None:
        a.Mi, a.Mi_sn, a.Mi_sm = Mi.data_ptr(), _bstride(Mi, 0), _bstride(Mi, 1)
    a.rf, a.rf_sn, a.rf_sx, a.rf_st = rf.data_ptr(), _bstride(rf, 0), rf.stride(1), rf.stride(2)
    a.rf_sc = rf.stride(3) if rf.ndim == 4 else 0
    a.gr, a.gr_sn, a.gr_sx, a.gr_st = gr.data_ptr(), _bstride(gr, 0), gr.stride(1), gr.stride(2)
    a.loc, a.loc_sn, a.loc_sm = loc.data_ptr(), _bstride(loc, 0), _bstride(loc, 1)
    if b1 is not None:
        a.b1, a.b1_sn, a.b1_sm = b1.data_ptr(), _bstride(b1, 0), _bstride(b1, 1)
    a.df = _param(df, N, nM)
    a.T1, a.T2 = _param(T1, N, nM), _param(T2, N, nM)
    a.gamma = _param(gamma, N, nM)
    a.dt = _param(dt, N, nM, per_batch_only=True)


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _fill_readout(a, nRx: int, rx: Optional[Tensor]):
    """The readout fields: nRx receive coils, the map rx (N|1, nM, 2, nRx) with inner (2, nRx) contiguous, or None (c = 1)."""
    a.nRx = nRx
    if rx is not None:
        assert rx.shape[3] == nRx, 'rx and nRx disagree on the receive coils'
        a.rx, a.rx_sn, a.rx_sm = rx.data_ptr(), _bstride(rx, 0), _bstride(rx, 1)


def _impl_blochsim_fused_fwd(Mi: Tensor, rf: Tensor, gr: Tensor, loc: Tensor, df: Optional[Tensor], b1: Optional[Tensor],
                             T1: Optional[Tensor], T2: Optional[Tensor], gamma: Tensor, dt: Tensor, K: int, flags: int,
                             every: int, nRx: int = 0, rx: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """-> (Mo (N,nM,3), out, ckpt, wave): final magnetisation, the option's output, K-step checkpoints, packed waveform.
    - every > 0, nRx == 0: out = Mt (N, nR, 3, nM), nR = nT // every: the state after (r+1)*every steps, lab frame.
    - nRx >= 1 (needs every > 0): out = S (N, 2, nR, nRx), the signal of those states summed over spins,
      S[n, :, r, k] = sum_i rx[n, i, :, k] * (Mx + i My)[n, i] (complex product; rx None: 1, with nRx = 1).
    - otherwise out is (0,)."""
    L = _cabi.lib()
    a = _cabi.FusedArgs()
    _fill_common(a, Mi, rf, gr, loc, df, b1, T1, T2, gamma, dt, K, flags)
    kw = {'dtype': Mi.dtype, 'device': Mi.device}
    Mo = torch.empty((a.N, a.nM, 3), **kw)
    ckpt = torch.empty(L.mrphy_fused_ckpt_elems(a), **kw)
    wave = torch.empty(L.mrphy_fused_wave_elems(a), **kw)
    a.Mo, a.ckpt, a.wave = Mo.data_ptr(), ckpt.data_ptr(), wave.data_ptr()
    if every:
        a.every, a.nR = every, a.nT // every
    if nRx:
        _fill_readout(a, nRx, rx)
        out = torch.empty((a.N, 2, a.nR, nRx), **kw)
        with torch.cuda.device(Mi.device):        # the workspace is sized from THIS device's SM count
            work = torch.empty(L.mrphy_fused_readout_elems(a), **kw)
        a.S, a.S_work = out.data_ptr(), work.data_ptr()
    else:
        out = torch.empty((a.N, a.nR, 3, a.nM) if every else (0,), **kw)
        if every:
            a.Mt = out.data_ptr()
    with torch.cuda.device(Mi.device):
        _cabi.check(L.mrphy_blochsim_fused_fwd(a, _stream()), 'blochsim_fused_fwd')
    _cabi.count_launches()
    return Mo, out, ckpt, wave


def _fake_blochsim_fused_fwd(Mi, rf, gr, loc, df, b1, T1, T2, gamma, dt, K, flags, every, nRx=0, rx=None):
    N, nM, nT = loc.shape[0], loc.shape[1], rf.shape[2]
    chunks = (nT + K - 1) // K
    nc = 1 if b1 is None else (rf.shape[3] if rf.ndim == 4 else 1)
    NC = next(c for c in (1, 2, 4, 8, 16) if nc <= c)           # coils held in registers (csrc: make_plan)
    W = 2 * NC + 3
    WS = (W + 3) // 4 * 4 if W * Mi.element_size() > 44 else W  # csrc: WaveLayout (step-major staging for many rows)
    chunk = WS * ((K + 3) // 4 * 4)
    if Mi.element_size() == 4 and NC >= 4 and K <= TC_K_MAX and os.environ.get('MRPHY_B200_TC', '1')[:1] != '0':
        chunk = max(chunk, ((K + 7) // 8 * 8) * (16 * (NC // 2) + 3))   # csrc: TcLayout (tensor-core operand tiles + gr rows)
    out = (N, 2, nT // every, nRx) if nRx else ((N, nT // every, 3, nM) if every else (0,))
    return (Mi.new_empty((N, nM, 3)), Mi.new_empty(out), Mi.new_empty((max(N * (chunks - 1) * 3 * nM, 1),)),
            Mi.new_empty((N * chunks * chunk,)))


def _impl_blochsim_fused_bwd(gMo: Tensor, gMt: Optional[Tensor], Mo: Tensor, ckpt: Tensor, wave: Tensor, rf: Tensor,
                             gr: Tensor, loc: Tensor, df: Optional[Tensor], b1: Optional[Tensor], T1: Optional[Tensor],
                             T2: Optional[Tensor], gamma: Tensor, dt: Tensor, K: int, flags: int, every: int, want_loc: bool,
                             want_sz: bool, want_b1: bool, rho: Optional[Tensor], theta: Optional[Tensor],
                             rfmax: Optional[Tensor], ts: Optional[Tensor], smax: Optional[Tensor], ddt: Optional[Tensor],
                             rf_kind: int, gr_kind: int, nRx: int = 0, rx: Optional[Tensor] = None, want_rx: bool = False):
    """-> (gMi (N,nM,3) or empty, flat, gloc, gsz, gb1, grho, gtheta, gts, grx); every output not asked for is (0,).
    flat = [dL/drf like rf (absent with FLAG_SKIP_GRF) | dL/dgr (N,3,nT) (absent with FLAG_SKIP_GGR) | GRAD_TAIL spare
    elements, zero]; `split_wave_grads` cuts the views.  Options:
    - every > 0, nRx == 0: the backward of a recording forward; gMt = dL/dMt (N, nR, 3, nM) contiguous on top of dL/dMo.
    - want_loc / want_sz / want_b1: the per-spin sums over time of dL/dBeff, formed inside the backward kernel without the
      dense field: gloc (N,nM,3) = sum_t gr*gBz, gsz (N,nM) = sum_t gBz, gb1 (N,nM,2,nC) -- the outputs of
      rfgr2beff_spin_grads.  want_b1 needs b1.
    - rf_kind / gr_kind > 0: (dL/drho, dL/dtheta, dL/dts) of the re-parametrisation (rho, theta, rfmax) -> rf,
      (ts, smax, ddt) -> gr, evaluated in the tail of the gradient epilogue: no launch of its own.  Combines with neither
      of the others.
    - nRx >= 1: the backward of a readout forward with the same every, nRx, rx; gMt = dL/dS (N, 2, nR, nRx) contiguous on
      top of dL/dMo, and with want_rx grx = dL/drx (N, nM, 2, nRx).  Combines with the per-spin gradients."""
    L = _cabi.lib()
    a = _cabi.FusedArgs()
    _fill_common(a, None, rf, gr, loc, df, b1, T1, T2, gamma, dt, K, flags)
    kw = {'dtype': Mo.dtype, 'device': Mo.device}
    need_gmi = bool(flags & _cabi.FLAG_NEED_GMI)
    gMi = torch.empty((a.N, a.nM, 3) if need_gmi else (0,), **kw)
    want_rf, want_gr = not flags & _cabi.FLAG_SKIP_GRF, not flags & _cabi.FLAG_SKIP_GGR
    # ONE flat buffer [dL/drf | dL/dgr | GRAD_TAIL spare elements]: both gradients are views of it, so a sharded run sums
    # them over ranks with a single in-place all-reduce of the buffer (mrphy.parallel), the spare tail carrying the loss
    n_rf, n_gr = (rf.numel() if want_rf else 0), (a.N * 3 * a.nT if want_gr else 0)
    flat = torch.empty(n_rf + n_gr + GRAD_TAIL, **kw)
    if want_rf or want_gr:
        a.flags |= _cabi.FLAG_ZERO_GRAD_TAIL       # the gradient epilogue zeroes the spare tail: no fill launch of its own
    else:
        flat.zero_()
    grf = flat[:n_rf].view(rf.shape) if want_rf else flat[:0]
    ggr = flat[n_rf:n_rf + n_gr].view(a.N, 3, a.nT) if want_gr else flat[:0]
    with torch.cuda.device(Mo.device):        # the workspace is sized from THIS device's SM count
        partials = torch.empty(L.mrphy_fused_partial_elems(a), **kw)
    a.Mo, a.ckpt, a.wave = Mo.data_ptr(), ckpt.data_ptr(), wave.data_ptr()
    a.gMo, a.gMo_sn, a.gMo_sm = gMo.data_ptr(), _bstride(gMo, 0), _bstride(gMo, 1)
    a.gMi, a.grf, a.ggr, a.partials = (gMi.data_ptr() if need_gmi else None), (grf.data_ptr() if want_rf else None), \
        (ggr.data_ptr() if want_gr else None), partials.data_ptr()
    gloc = gsz = gb1 = grho = gtheta = gts = grx = flat[:0]
    if every:
        a.every, a.nR = every, a.nT // every
    if nRx:
        _fill_readout(a, nRx, rx)
        a.gS = gMt.data_ptr()
        if want_rx:
            grx = torch.empty((a.N, a.nM, 2, nRx), **kw)
            a.grx = grx.data_ptr()
    elif every and gMt is not None:
        a.gMt = gMt.data_ptr()
    if want_loc or want_sz or want_b1:
        e = lambda shape, on: torch.empty(shape if on else (0,), **kw)
        gloc, gsz, gb1 = e((a.N, a.nM, 3), want_loc), e((a.N, a.nM), want_sz), e((a.N, a.nM, 2, a.nC), want_b1)
        a.gloc, a.gsz, a.gb1 = (gloc.data_ptr() if want_loc else None), (gsz.data_ptr() if want_sz else None), \
            (gb1.data_ptr() if want_b1 else None)
    d = None                                  # the ReparamArgs a.design points to: alive until the call returns
    if rf_kind or gr_kind:
        d, _ = _reparam_args(rho, theta, rfmax, ts, smax, ddt, rf_kind, gr_kind, True)
        if rf_kind:
            grho, gtheta = torch.empty(rho.shape, **kw), torch.empty(theta.shape, **kw)
            d.grho, d.gtheta = grho.data_ptr(), gtheta.data_ptr()
        if gr_kind:
            gts = torch.empty(ts.shape, **kw)
            d.gts = gts.data_ptr()
        a.design = ctypes.addressof(d)
    with torch.cuda.device(Mo.device):
        _cabi.check(L.mrphy_blochsim_fused_bwd(a, 1, _stream()), 'blochsim_fused_bwd')
    _cabi.count_launches()
    return gMi, flat, gloc, gsz, gb1, grho, gtheta, gts, grx


def _fake_blochsim_fused_bwd(gMo, gMt, Mo, ckpt, wave, rf, gr, loc, df, b1, T1, T2, gamma, dt, K, flags, every, want_loc,
                             want_sz, want_b1, rho, theta, rfmax, ts, smax, ddt, rf_kind, gr_kind, nRx=0, rx=None,
                             want_rx=False):
    n = (0 if flags & _cabi.FLAG_SKIP_GRF else rf.numel()) + (0 if flags & _cabi.FLAG_SKIP_GGR else rf.shape[0] * 3 * rf.shape[2])
    N, nM, nC = loc.shape[0], loc.shape[1], (rf.shape[3] if rf.ndim == 4 else 1)
    e = lambda shape, on: Mo.new_empty(shape if on else (0,))
    return (e(Mo.shape, flags & _cabi.FLAG_NEED_GMI), Mo.new_empty((n + GRAD_TAIL,)), e((N, nM, 3), want_loc),
            e((N, nM), want_sz), e((N, nM, 2, nC), want_b1), e(rho.shape if rf_kind else (), rf_kind),
            e(theta.shape if rf_kind else (), rf_kind), e(ts.shape if gr_kind else (), gr_kind),
            e((N, nM, 2, nRx), nRx and want_rx))


GRAD_TAIL = 4      # spare elements behind the waveform gradients (16-byte granule); [0] is where `parallel` puts the loss


def split_wave_grads(flat: Tensor, rf: Tensor, flags: int):
    """(dL/drf, dL/dgr) as views of the backward's flat buffer (None where skipped)."""
    N, nT = rf.shape[0], rf.shape[2]
    n_rf = 0 if flags & _cabi.FLAG_SKIP_GRF else rf.numel()
    n_gr = 0 if flags & _cabi.FLAG_SKIP_GGR else N * 3 * nT
    return (flat[:n_rf].view(rf.shape) if n_rf else None), (flat[n_rf:n_rf + n_gr].view(N, 3, nT) if n_gr else None)


def _fused_grads(ctx, want, gMo, Mo, ckpt, wave, rf, gr, loc, df, b1, T1, T2, gamma, dt, gMt=None, every=0,
                 spin=(False, False, False), design=(None,) * 6 + (0, 0), readout=(0, None, False)):
    """The fused backward of a forward run with ctx.K, ctx.flags.  want = (dL/dMi, dL/drf, dL/dgr) wanted: the rows of the
    spin reduction of the others are not even formed.  -> (gMi or None, grf, ggr, gloc, gsz, gb1, grho, gtheta, gts, grx);
    with readout = (nRx, rx, want_rx), nRx >= 1, gMt is dL/dS of a readout forward."""
    if gMo is None:
        gMo = torch.zeros_like(Mo)
    if gMo.stride(-1) != 1 or gMo.dtype != Mo.dtype:
        gMo = gMo.to(Mo.dtype).contiguous()
    flags = ctx.flags | (_cabi.FLAG_NEED_GMI if want[0] else 0) | (0 if want[1] else _cabi.FLAG_SKIP_GRF) | \
        (0 if want[2] else _cabi.FLAG_SKIP_GGR)
    gMi, flat, *rest = blochsim_fused_bwd(gMo, gMt, Mo, ckpt, wave, rf, gr, loc, df, b1, T1, T2, gamma, dt, ctx.K, flags,
                                          every, *spin, *design, *readout)
    return (gMi if want[0] else None, *split_wave_grads(flat, rf, flags), *rest)


def _fused_setup(ctx, inputs, output):
    Mi, rf, gr, loc, df, b1, T1, T2, gamma, dt, K, flags, every, nRx, rx = inputs
    Mo, _Mt, ckpt, wave = output
    ctx.K, ctx.flags, ctx.every, ctx.nRx = K, flags, every, nRx
    opt = (df, b1, T1, T2, rx)
    ctx.has = [x is not None for x in opt]
    ctx.save_for_backward(Mo, ckpt, wave, rf, gr, loc, gamma, dt, *[x for x in opt if x is not None])
    if every:
        ctx.set_materialize_grads(False)      # a loss that ignores Mt / S (or M) hands None for it, not a tensor of zeros


def _param_2d(x: Tensor) -> Tensor:
    """A per-spin constant viewed the way `_param` reads it: (N|1, nM|1) from that, (N|1,) per batch entry, () or trailing
    singleton dims."""
    v = x
    while v.ndim > 2 and v.shape[-1] == 1:
        v = v[..., 0]
    return v.reshape(1, 1) if v.ndim == 0 else (v[:, None] if v.ndim == 1 else v)


def _as_param_grad(g: Tensor, x: Tensor) -> Tensor:
    """A per-spin gradient (N,nM) reduced to the shape and dtype of the op input `x` (see `_param_2d`)."""
    return g.sum_to_size(_param_2d(x).shape).reshape(x.shape).to(x.dtype)


def _fused_backward(ctx, gMo, gMt, _gckpt, _gwave):
    """With no gradient on Mt / S (or neither option) the backward without them (same kernels, same bits); else the REC or
    readout backward, with dL/dMo = 0 when the loss ignores M."""
    Mo, ckpt, wave, rf, gr, loc, gamma, dt, *opt = ctx.saved_tensors
    opt = list(opt)
    df, b1, T1, T2, rx = (opt.pop(0) if h else None for h in ctx.has)
    need = ctx.needs_input_grad           # (trailing inputs left at their defaults have no entry)
    # per-spin gradients (inputs loc, df, b1, gamma): γ reaches the loss only through Bz += df/γ, so without df it has none
    want_loc, want_b1 = bool(need[3]), bool(need[5] and b1 is not None)
    want_sz = df is not None and bool(need[4] or need[8])
    want_rx = rx is not None and bool(need[14]) and gMt is not None
    if not (any(need[0:3]) or want_loc or want_sz or want_b1 or want_rx):
        return (None,) * len(need)
    every = ctx.every if gMt is not None else 0
    if every and (gMt.dtype != Mo.dtype or not gMt.is_contiguous()):
        # dL/dMt (dL/dS) in the kernel's layout (N, nR, 3, nM) ((N, 2, nR, nRx)) and dtype: a loss formed elementwise from the
        # view the caller got hands its gradient back in that layout already; anything else costs this one copy
        gMt = torch.empty(gMt.shape, dtype=Mo.dtype, device=Mo.device).copy_(gMt)
    gMi, grf, ggr, gloc, gsz, gb1, *_, grx = _fused_grads(ctx, need[0:3], gMo, Mo, ckpt, wave, rf, gr, loc, df, b1, T1, T2,
                                                          gamma, dt, gMt if every else None, every,
                                                          (want_loc, want_sz, want_b1),
                                                          readout=(ctx.nRx if every else 0, rx, want_rx))
    gdf = ggam = None
    if want_sz:     # ∂Δf = gsz/γ, ∂γ = -gsz·Δf/γ² (the chain rule of Bz += Δf/γ, beffective.py:142)
        gam2, df2 = _param_2d(gamma), _param_2d(df)
        if need[4]:
            gdf = _as_param_grad(gsz / gam2, df)
        if need[8]:
            ggam = _as_param_grad(-gsz * df2 / (gam2 * gam2), gamma)
    return (gMi, grf, ggr, gloc if want_loc else None, gdf, gb1 if want_b1 else None, None, None, ggam, None, None, None,
            None, None, grx.sum_to_size(rx.shape) if want_rx else None)


# ------------------------------------------------------------------------------------------------
# explicit-field ops: sims.BlochSim.forward / backward on a dense Beff (sims.py:31-269)
def _fill_beff(a, Mi, Beff, T1, T2, gamma, dt, K, flags):
    N, nM, nT = Beff.shape[0], Beff.shape[1], Beff.shape[2]
    a.dtype = _cabi.MRPHY_F64 if Beff.dtype == torch.float64 else _cabi.MRPHY_F32
    a.flags, a.N, a.nM, a.nT, a.K = flags, N, nM, nT, K
    if Mi is not None:
        a.Mi, a.Mi_sn, a.Mi_sm = Mi.data_ptr(), _bstride(Mi, 0), _bstride(Mi, 1)
    a.Beff, a.B_sn, a.B_sm, a.B_st = Beff.data_ptr(), _bstride(Beff, 0), _bstride(Beff, 1), 3
    a.T1, a.T2 = _param(T1, N, nM), _param(T2, N, nM)
    a.gamma = _param(gamma, N, nM)
    a.dt = _param(dt, N, nM, per_batch_only=True)


def _impl_blochsim_beff_fwd(Mi: Tensor, Beff: Tensor, T1: Optional[Tensor], T2: Optional[Tensor], gamma: Tensor,
                      dt: Tensor, K: int, flags: int) -> Tuple[Tensor, Tensor]:
    """Mi (N,nM,3), Beff (N,nM,nT,3) -> (Mo (N,nM,3), ckpt)."""
    L = _cabi.lib()
    a = _cabi.BeffArgs()
    _fill_beff(a, Mi, Beff, T1, T2, gamma, dt, K, flags)
    kw = {'dtype': Mi.dtype, 'device': Mi.device}
    Mo = torch.empty((a.N, a.nM, 3), **kw)
    ckpt = torch.empty(L.mrphy_beff_ckpt_elems(a), **kw)
    a.Mo, a.ckpt = Mo.data_ptr(), ckpt.data_ptr()
    with torch.cuda.device(Mi.device):
        _cabi.check(L.mrphy_blochsim_beff_fwd(a, _stream()), 'blochsim_beff_fwd')
    _cabi.count_launches()
    return Mo, ckpt


def _fake_blochsim_beff_fwd(Mi, Beff, T1, T2, gamma, dt, K, flags):
    N, nM, nT = Beff.shape[0], Beff.shape[1], Beff.shape[2]
    return Mi.new_empty((N, nM, 3)), Mi.new_empty((max(N * ((nT - 1) // K) * 3 * nM, 1),))


def _impl_blochsim_beff_bwd(gMo: Tensor, Mo: Tensor, ckpt: Tensor, Beff: Tensor, T1: Optional[Tensor],
                      T2: Optional[Tensor], gamma: Tensor, dt: Tensor, K: int, flags: int) -> Tuple[Tensor, Tensor]:
    """-> (gMi (N,nM,3) or empty, gBeff (N,nM,nT,3) or empty)."""
    L = _cabi.lib()
    a = _cabi.BeffArgs()
    _fill_beff(a, None, Beff, T1, T2, gamma, dt, K, flags)
    kw = {'dtype': Mo.dtype, 'device': Mo.device}
    need_gmi, need_gb = bool(flags & _cabi.FLAG_NEED_GMI), bool(flags & _cabi.FLAG_NEED_GBEFF)
    gMi = torch.empty((a.N, a.nM, 3) if need_gmi else (0,), **kw)
    gB = torch.empty((a.N, a.nM, a.nT, 3) if need_gb else (0,), **kw)
    a.Mo, a.ckpt = Mo.data_ptr(), ckpt.data_ptr()
    a.gMo, a.gMo_sn, a.gMo_sm = gMo.data_ptr(), _bstride(gMo, 0), _bstride(gMo, 1)
    a.gMi = gMi.data_ptr() if need_gmi else None
    a.gBeff = gB.data_ptr() if need_gb else None
    with torch.cuda.device(Mo.device):
        _cabi.check(L.mrphy_blochsim_beff_bwd(a, _stream()), 'blochsim_beff_bwd')
    _cabi.count_launches()
    return gMi, gB


def _fake_blochsim_beff_bwd(gMo, Mo, ckpt, Beff, T1, T2, gamma, dt, K, flags):
    return (Mo.new_empty(Mo.shape if flags & _cabi.FLAG_NEED_GMI else (0,)),
            Mo.new_empty(Beff.shape if flags & _cabi.FLAG_NEED_GBEFF else (0,)))


def beff_ckpt_interval(K: int) -> int:
    """The explicit-field kernels take K in {1..32} or 64 (tile-aligned)."""
    return K if K <= 32 else (64 if K >= 64 else 32)


# ------------------------------------------------------------------------------------------------
# stand-alone operators: rfgr2beff, beff2ab (+ adjoint), beff2uphi (+ adjoint), freeprec
def _rfgr2beff_args(rf, gr, loc, df, b1, gamma):
    a = _cabi.RfGr2BeffArgs()
    N, nM, nT = loc.shape[0], loc.shape[1], rf.shape[2]
    a.dtype = _cabi.MRPHY_F64 if loc.dtype == torch.float64 else _cabi.MRPHY_F32
    a.flags = _cabi.FLAG_RF_COIL_DIM if rf.ndim == 4 else 0
    a.N, a.nM, a.nT, a.nC = N, nM, nT, (rf.shape[3] if rf.ndim == 4 else 1)
    a.rf, a.rf_sn, a.rf_sx, a.rf_st = rf.data_ptr(), _bstride(rf, 0), rf.stride(1), rf.stride(2)
    a.rf_sc = rf.stride(3) if rf.ndim == 4 else 0
    a.gr, a.gr_sn, a.gr_sx, a.gr_st = gr.data_ptr(), _bstride(gr, 0), gr.stride(1), gr.stride(2)
    a.loc, a.loc_sn, a.loc_sm = loc.data_ptr(), _bstride(loc, 0), _bstride(loc, 1)
    if b1 is not None:
        a.b1, a.b1_sn, a.b1_sm = b1.data_ptr(), _bstride(b1, 0), _bstride(b1, 1)
    a.df, a.gamma = _param(df, N, nM), _param(gamma, N, nM)
    return a


def _impl_rfgr2beff(rf: Tensor, gr: Tensor, loc: Tensor, df: Optional[Tensor], b1: Optional[Tensor],
                   gamma: Tensor) -> Tensor:
    """rf (N,2,nT[,nC]), gr (N,3,nT), loc (N,nM,3), df (N|1,nM|1), b1 (N,nM,2,nC) -> Beff (N,nM,nT,3)."""
    L = _cabi.lib()
    a = _rfgr2beff_args(rf, gr, loc, df, b1, gamma)
    out = torch.empty((a.N, a.nM, a.nT, 3), dtype=loc.dtype, device=loc.device)
    a.Beff = out.data_ptr()
    with torch.cuda.device(loc.device):
        _cabi.check(L.mrphy_rfgr2beff(a, _stream()), 'rfgr2beff')
    _cabi.count_launches()
    return out


def _impl_rfgr2beff_bwd(gB: Tensor, rf: Tensor, gr: Tensor, loc: Tensor, b1: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """gB (N,nM,nT,3) contiguous -> (grf like rf, ggr (N,3,nT)): the sums over spins of rfgr2beff's chain rule."""
    L = _cabi.lib()
    a = _rfgr2beff_args(rf, gr, loc, None, b1, None)
    kw = {'dtype': loc.dtype, 'device': loc.device}
    grf, ggr = torch.empty(rf.shape, **kw), torch.empty((a.N, 3, a.nT), **kw)
    part = torch.empty(L.mrphy_rfgr2beff_partial_elems(a), **kw)
    a.gBeff, a.grf, a.ggr, a.partials = gB.data_ptr(), grf.data_ptr(), ggr.data_ptr(), part.data_ptr()
    with torch.cuda.device(loc.device):
        _cabi.check(L.mrphy_rfgr2beff_bwd(a, _stream()), 'rfgr2beff_bwd')
    _cabi.count_launches()
    return grf, ggr


def _impl_rfgr2beff_spin_grads(gB: Tensor, rf: Tensor, gr: Tensor, want_loc: bool, want_b1: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """gB (N,nM,nT,3) contiguous -> (gloc (N,nM,3) = sum_t gr*gBz, gsz (N,nM) = sum_t gBz, gb1 (N,nM,2,nC)): the per-spin
    (time-summed) half of rfgr2beff's chain rule in one pass over gB; unwanted outputs come back empty."""
    L = _cabi.lib()
    a = _cabi.RfGr2BeffArgs()
    N, nM, nT = gB.shape[0], gB.shape[1], gB.shape[2]
    nC = rf.shape[3] if rf.ndim == 4 else 1
    a.dtype = _cabi.MRPHY_F64 if gB.dtype == torch.float64 else _cabi.MRPHY_F32
    a.flags = _cabi.FLAG_RF_COIL_DIM if rf.ndim == 4 else 0
    a.N, a.nM, a.nT, a.nC = N, nM, nT, nC
    a.rf, a.rf_sn, a.rf_sx, a.rf_st = rf.data_ptr(), _bstride(rf, 0), rf.stride(1), rf.stride(2)
    a.rf_sc = rf.stride(3) if rf.ndim == 4 else 0
    a.gr, a.gr_sn, a.gr_sx, a.gr_st = gr.data_ptr(), _bstride(gr, 0), gr.stride(1), gr.stride(2)
    kw = {'dtype': gB.dtype, 'device': gB.device}
    gloc = torch.empty((N, nM, 3) if want_loc else (0,), **kw)
    gsz = torch.empty((N, nM), **kw)
    gb1 = torch.empty((N, nM, 2, nC) if want_b1 else (0,), **kw)
    a.gBeff, a.gsz = gB.data_ptr(), gsz.data_ptr()
    if want_loc:
        a.gloc = gloc.data_ptr()
    if want_b1:
        a.gb1 = gb1.data_ptr()
    with torch.cuda.device(gB.device):
        _cabi.check(L.mrphy_rfgr2beff_spin_grads(a, _stream()), 'rfgr2beff_spin_grads')
    _cabi.count_launches()
    return gloc, gsz, gb1


def _fake_rfgr2beff_spin_grads(gB, rf, gr, want_loc, want_b1):
    N, nM = gB.shape[0], gB.shape[1]
    nC = rf.shape[3] if rf.ndim == 4 else 1
    return (gB.new_empty((N, nM, 3) if want_loc else (0,)), gB.new_empty((N, nM)),
            gB.new_empty((N, nM, 2, nC) if want_b1 else (0,)))


def _fake_rfgr2beff_bwd(gB, rf, gr, loc, b1):
    return rf.new_empty(rf.shape), gr.new_empty((loc.shape[0], 3, rf.shape[2]))


def _fake_rfgr2beff(rf, gr, loc, df, b1, gamma):
    return loc.new_empty((loc.shape[0], loc.shape[1], rf.shape[2], 3))


def _beff2ab_args(beff, E1, E2, gamma, dt, K, flags):
    a = _cabi.Beff2abArgs()
    N, nM, nT = beff.shape[0], beff.shape[1], beff.shape[2]
    a.dtype = _cabi.MRPHY_F64 if beff.dtype == torch.float64 else _cabi.MRPHY_F32
    a.flags, a.N, a.nM, a.nT, a.K = flags, N, nM, nT, K
    a.Beff, a.B_sn, a.B_sm = beff.data_ptr(), _bstride(beff, 0), _bstride(beff, 1)
    a.E1, a.E2, a.gamma = _param(E1, N, nM), _param(E2, N, nM), _param(gamma, N, nM)
    a.dt = _param(dt, N, nM, per_batch_only=True)
    return a


def _impl_beff2ab(beff: Tensor, E1: Tensor, E2: Tensor, gamma: Tensor, dt: Tensor, K: int,
                  flags: int) -> Tuple[Tensor, Tensor, Tensor]:
    """beff (N,nM,nT,3) -> A (N,nM,3,3), B (N,nM,3), ckpt; E1/E2/gamma broadcastable to (N,nM), dt () or (N|1,).
    K > 0 also stores [A|B] every K steps for the adjoint; K = 0: forward only (ckpt is empty)."""
    L = _cabi.lib()
    a = _beff2ab_args(beff, E1, E2, gamma, dt, K, flags)
    kw = {'dtype': beff.dtype, 'device': beff.device}
    A, B = torch.empty((a.N, a.nM, 3, 3), **kw), torch.empty((a.N, a.nM, 3), **kw)
    ckpt = torch.empty(L.mrphy_beff2ab_ckpt_elems(a) if K > 0 else 0, **kw)
    a.A, a.B = A.data_ptr(), B.data_ptr()
    if K > 0:
        a.ckpt = ckpt.data_ptr()
    with torch.cuda.device(beff.device):
        _cabi.check(L.mrphy_beff2ab(a, _stream()), 'beff2ab')
    _cabi.count_launches()
    return A, B, ckpt


def _fake_beff2ab(beff, E1, E2, gamma, dt, K, flags):
    N, nM, nT = beff.shape[:3]
    return (beff.new_empty((N, nM, 3, 3)), beff.new_empty((N, nM, 3)),
            beff.new_empty((max(N * ((nT - 1) // K) * 12 * nM, 1) if K > 0 else 0,)))


def _impl_beff2ab_bwd(gA: Tensor, gB: Tensor, A: Tensor, B: Tensor, ckpt: Tensor, beff: Tensor, E1: Tensor, E2: Tensor,
                      gamma: Tensor, dt: Tensor, K: int, flags: int) -> Tuple[Tensor, Tensor]:
    """-> gbeff (N,nM,nT,3), gP (N,nM,3) = per-spin [dL/dE1, dL/dE2, dL/d(2*pi*gamma*dt)]."""
    L = _cabi.lib()
    a = _beff2ab_args(beff, E1, E2, gamma, dt, K, flags)
    kw = {'dtype': beff.dtype, 'device': beff.device}
    gbeff, gP = torch.empty((a.N, a.nM, a.nT, 3), **kw), torch.empty((a.N, a.nM, 3), **kw)
    a.A, a.B, a.ckpt = A.data_ptr(), B.data_ptr(), ckpt.data_ptr()
    a.gA, a.gB, a.gBeff, a.gP = gA.data_ptr(), gB.data_ptr(), gbeff.data_ptr(), gP.data_ptr()
    with torch.cuda.device(beff.device):
        _cabi.check(L.mrphy_beff2ab_bwd(a, _stream()), 'beff2ab_bwd')
    _cabi.count_launches()
    return gbeff, gP


def _fake_beff2ab_bwd(gA, gB, A, B, ckpt, beff, E1, E2, gamma, dt, K, flags):
    return beff.new_empty(beff.shape), beff.new_empty(beff.shape[:2] + (3,))


def _impl_beff2uphi(beff: Tensor, g: Tensor) -> Tuple[Tensor, Tensor]:
    """beff (N,nM,3), g broadcastable to (N,nM) -> U (N,nM,3), Phi (N,nM)."""
    L = _cabi.lib()
    a = _cabi.Beff2uphiArgs()
    N, nM = beff.shape[0], beff.shape[1]
    a.dtype = _cabi.MRPHY_F64 if beff.dtype == torch.float64 else _cabi.MRPHY_F32
    a.N, a.nM = N, nM
    a.beff, a.b_sn, a.b_sm = beff.data_ptr(), _bstride(beff, 0), _bstride(beff, 1)
    a.g = _param(g, N, nM)
    U, Phi = torch.empty((N, nM, 3), dtype=beff.dtype, device=beff.device), torch.empty((N, nM), dtype=beff.dtype, device=beff.device)
    a.U, a.Phi = U.data_ptr(), Phi.data_ptr()
    with torch.cuda.device(beff.device):
        _cabi.check(L.mrphy_beff2uphi(a, _stream()), 'beff2uphi')
    _cabi.count_launches()
    return U, Phi


def _fake_beff2uphi(beff, g):
    return beff.new_empty(beff.shape), beff.new_empty(beff.shape[:2])


def _impl_beff2uphi_bwd(gU: Optional[Tensor], gPhi: Optional[Tensor], beff: Tensor, g: Tensor) -> Tuple[Tensor, Tensor]:
    """-> gbeff (N,nM,3), gg (N,nM) = per-spin dL/dg."""
    L = _cabi.lib()
    a = _cabi.Beff2uphiArgs()
    N, nM = beff.shape[0], beff.shape[1]
    a.dtype = _cabi.MRPHY_F64 if beff.dtype == torch.float64 else _cabi.MRPHY_F32
    a.adjoint, a.N, a.nM = 1, N, nM
    a.beff, a.b_sn, a.b_sm = beff.data_ptr(), _bstride(beff, 0), _bstride(beff, 1)
    a.g = _param(g, N, nM)
    gbeff, gg = torch.empty((N, nM, 3), dtype=beff.dtype, device=beff.device), torch.empty((N, nM), dtype=beff.dtype, device=beff.device)
    if gU is not None:
        a.gU = gU.data_ptr()
    if gPhi is not None:
        a.gPhi = gPhi.data_ptr()
    a.gbeff, a.gg = gbeff.data_ptr(), gg.data_ptr()
    with torch.cuda.device(beff.device):
        _cabi.check(L.mrphy_beff2uphi(a, _stream()), 'beff2uphi_bwd')
    _cabi.count_launches()
    return gbeff, gg


def _fake_beff2uphi_bwd(gU, gPhi, beff, g):
    return beff.new_empty(beff.shape), beff.new_empty(beff.shape[:2])


def _impl_freeprec(Mi: Tensor, dur: Tensor, T1: Optional[Tensor], T2: Optional[Tensor], df: Optional[Tensor],
                  adjoint: bool) -> Tensor:
    """Mi (N,nM,3) -> Mo (N,nM,3); with adjoint=True applies the transposed map to a gradient."""
    L = _cabi.lib()
    a = _cabi.FreePrecArgs()
    N, nM = Mi.shape[0], Mi.shape[1]
    a.dtype = _cabi.MRPHY_F64 if Mi.dtype == torch.float64 else _cabi.MRPHY_F32
    a.adjoint, a.N, a.nM = int(adjoint), N, nM
    a.Mi, a.Mi_sn, a.Mi_sm = Mi.data_ptr(), _bstride(Mi, 0), _bstride(Mi, 1)
    a.dur = _param(dur, N, nM, per_batch_only=True)
    a.T1, a.T2, a.df = _param(T1, N, nM), _param(T2, N, nM), _param(df, N, nM)
    Mo = torch.empty((N, nM, 3), dtype=Mi.dtype, device=Mi.device)
    a.Mo = Mo.data_ptr()
    with torch.cuda.device(Mi.device):
        _cabi.check(L.mrphy_freeprec(a, _stream()), 'freeprec')
    _cabi.count_launches()
    return Mo


def _fake_freeprec(Mi, dur, T1, T2, df, adjoint):
    return Mi.new_empty(Mi.shape)


def _reparam_args(rho, theta, rfmax, ts, smax, dt, rf_kind, gr_kind, adjoint):
    """Fill the C struct from (already validated, contiguous) tensors; returns (args, N, nT, nC, dtype, device)."""
    a = _cabi.ReparamArgs()
    lead = rho if rf_kind else ts
    N, nT = lead.shape[0], lead.shape[2]
    nC = rho.shape[3] if (rf_kind and rho.ndim == 4) else 1
    a.dtype = _cabi.MRPHY_F64 if lead.dtype == torch.float64 else _cabi.MRPHY_F32
    a.adjoint, a.N, a.nT, a.nC, a.rf_kind, a.gr_kind = int(adjoint), N, nT, nC, rf_kind, gr_kind
    if rf_kind:
        a.rho, a.theta = rho.data_ptr(), theta.data_ptr()
        v = rfmax.expand((N, nC))                      # (N|1, nC|1) -> strides, 0 where broadcast
        a.rfmax, a.rfmax_sn, a.rfmax_sc = v.data_ptr(), v.stride(0), v.stride(1)
    if gr_kind:
        a.ts = ts.data_ptr()
        if gr_kind != 2:
            v = smax.expand((N, 3))
            a.smax, a.smax_sn, a.smax_sx = v.data_ptr(), v.stride(0), v.stride(1)
        if gr_kind != 3:
            a.dt = _param(dt, N, 1, per_batch_only=True)
    return a, lead


def _impl_design_waveform(rho: Optional[Tensor], theta: Optional[Tensor], rfmax: Optional[Tensor], ts: Optional[Tensor],
                          smax: Optional[Tensor], dt: Optional[Tensor], rf_kind: int, gr_kind: int) -> Tuple[Tensor, Tensor]:
    """One launch: (rho, theta, rfmax) -> rf (N,2,nT[,nC]) and/or (ts|s, smax, dt) -> gr|s (N,3,nT); an absent half
    returns an empty tensor.  rfmax is (N|1, nC|1), smax (N|1, 3|1) (see utils._design_call)."""
    L = _cabi.lib()
    a, lead = _reparam_args(rho, theta, rfmax, ts, smax, dt, rf_kind, gr_kind, False)
    rf = torch.empty((rho.shape[0], 2) + tuple(rho.shape[2:]) if rf_kind else (0,), dtype=lead.dtype, device=lead.device)
    gr = torch.empty(ts.shape if gr_kind else (0,), dtype=lead.dtype, device=lead.device)
    a.rf, a.gr = rf.data_ptr(), gr.data_ptr()
    with torch.cuda.device(lead.device):
        _cabi.check(L.mrphy_design_waveform(a, _stream()), 'design_waveform')
    _cabi.count_launches()
    return rf, gr


def _fake_design_waveform(rho, theta, rfmax, ts, smax, dt, rf_kind, gr_kind):
    lead = rho if rf_kind else ts
    return (lead.new_empty((rho.shape[0], 2) + tuple(rho.shape[2:]) if rf_kind else (0,)),
            lead.new_empty(ts.shape if gr_kind else (0,)))


def _impl_design_waveform_bwd(grf: Optional[Tensor], ggr: Optional[Tensor], rho: Optional[Tensor], theta: Optional[Tensor],
                              rfmax: Optional[Tensor], ts: Optional[Tensor], smax: Optional[Tensor], dt: Optional[Tensor],
                              rf_kind: int, gr_kind: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Adjoint in one launch: (dL/drf, dL/dgr) -> (dL/drho, dL/dtheta, dL/dts); absent halves come back empty."""
    L = _cabi.lib()
    a, lead = _reparam_args(rho, theta, rfmax, ts, smax, dt, rf_kind, gr_kind, True)
    e = lambda like, on: torch.empty(like.shape if on else (0,), dtype=lead.dtype, device=lead.device)
    grho, gtheta, gts = e(rho if rf_kind else lead, rf_kind), e(theta if rf_kind else lead, rf_kind), e(ts if gr_kind else lead, gr_kind)
    if rf_kind:
        grf = grf.contiguous()
        a.grf, a.grho, a.gtheta = grf.data_ptr(), grho.data_ptr(), gtheta.data_ptr()
    if gr_kind:
        ggr = ggr.contiguous()
        a.ggr, a.gts = ggr.data_ptr(), gts.data_ptr()
    with torch.cuda.device(lead.device):
        _cabi.check(L.mrphy_design_waveform(a, _stream()), 'design_waveform (adjoint)')
    _cabi.count_launches()
    return grho, gtheta, gts


def _fake_design_waveform_bwd(grf, ggr, rho, theta, rfmax, ts, smax, dt, rf_kind, gr_kind):
    lead = rho if rf_kind else ts
    e = lambda like, on: lead.new_empty(like.shape if on else (0,))
    return e(rho if rf_kind else lead, rf_kind), e(theta if rf_kind else lead, rf_kind), e(ts if gr_kind else lead, gr_kind)


def _design_setup(ctx, inputs, output):
    rho, theta, rfmax, ts, smax, dt, rf_kind, gr_kind = inputs
    ctx.save_for_backward(rho, theta, rfmax, ts, smax, dt)
    ctx.kinds = (rf_kind, gr_kind)


def _design_backward(ctx, grf, ggr):
    rho, theta, rfmax, ts, smax, dt = ctx.saved_tensors
    rf_kind, gr_kind = ctx.kinds
    if rf_kind and grf is None:
        grf = torch.zeros((rho.shape[0], 2) + tuple(rho.shape[2:]), dtype=rho.dtype, device=rho.device)
    if gr_kind and ggr is None:
        ggr = torch.zeros_like(ts)
    grho, gtheta, gts = design_waveform_bwd_cuda(grf if rf_kind else None, ggr if gr_kind else None, rho, theta, rfmax, ts,
                                                 smax, dt, rf_kind, gr_kind)
    return (grho if rf_kind else None, gtheta if rf_kind else None, None, gts if gr_kind else None, None, None, None, None)


def _clamp_call(x: Tensor, lim: Tensor, eps: float, kind: int, g: Optional[Tensor]) -> Tensor:
    L = _cabi.lib()
    a = _cabi.ClampArgs()
    a.dtype = _cabi.MRPHY_F64 if x.dtype == torch.float64 else _cabi.MRPHY_F32
    a.adjoint, a.kind, a.N, a.nT = int(g is not None), kind, x.shape[0], x.shape[2]
    a.nC = x.shape[3] if (kind == 1 and x.ndim == 4) else 1
    v = lim.expand((x.shape[0], a.nC if kind == 1 else 3))            # (N|1, nC|1 or 3|1) -> strides, 0 where broadcast
    a.x, a.lim, a.lim_sn, a.lim_sc, a.eps = x.data_ptr(), v.data_ptr(), v.stride(0), v.stride(1), float(eps)
    out = torch.empty_like(x)
    a.out = out.data_ptr()
    if g is not None:
        a.g = g.data_ptr()
    with torch.cuda.device(x.device):
        _cabi.check(L.mrphy_clamp_waveform(a, _stream()), 'clamp_waveform')
    _cabi.count_launches()
    return out


def _impl_clamp_waveform(x: Tensor, lim: Tensor, eps: float, kind: int) -> Tensor:
    """kind 1: utils.rfclamp of rf (N,2,nT[,nC]) at rfmax `lim` (N|1, nC|1) - eps; kind 2: utils.sclamp of s (N,3,nT) at
    `lim` (N|1, 3|1).  x contiguous."""
    return _clamp_call(x, lim, eps, kind, None)


def _impl_clamp_waveform_bwd(g: Tensor, x: Tensor, lim: Tensor, eps: float, kind: int) -> Tensor:
    return _clamp_call(x, lim, eps, kind, g)


def _clamp_setup(ctx, inputs, output):
    x, lim, eps, kind = inputs
    ctx.save_for_backward(x, lim)
    ctx.eps, ctx.kind = eps, kind


def _clamp_backward(ctx, g):
    x, lim = ctx.saved_tensors
    return clamp_waveform_bwd_cuda(g.contiguous(), x, lim, ctx.eps, ctx.kind), None, None, None


def _impl_mask_copy(v: Tensor, idx: Tensor, inv: Tensor, fill_zero: bool) -> Tensor:
    """v (N,nIn,inner) contiguous, idx (nOut,) int64 -> out[n,j] = v[n,idx[j]], rows with idx[j] < 0 are NaN (or 0).
    ``inv`` (nIn,) is the inverse map; only the backward uses it."""
    L = _cabi.lib()
    a = _cabi.MaskArgs()
    n_out = idx.numel()
    a.dtype = _cabi.MRPHY_F64 if v.dtype == torch.float64 else _cabi.MRPHY_F32
    a.N, a.fill_zero, a.nOut, a.nIn, a.inner = v.shape[0], int(fill_zero), n_out, v.shape[1], v.shape[2]
    out = torch.empty((v.shape[0], n_out, v.shape[2]), dtype=v.dtype, device=v.device)
    a.idx, a.inp, a.out = idx.data_ptr(), v.data_ptr(), out.data_ptr()
    with torch.cuda.device(v.device):
        _cabi.check(L.mrphy_mask_copy(a, _stream()), 'mask_copy')
    _cabi.count_launches()
    return out


def _fake_mask_copy(v, idx, inv, fill_zero):
    return v.new_empty((v.shape[0], idx.numel(), v.shape[2]))


def _mask_setup(ctx, inputs, output):
    v, idx, inv, fill_zero = inputs
    ctx.save_for_backward(idx, inv)


def _mask_backward(ctx, g):
    # the transposed map of a gather with distinct sources is the gather with the inverse index, zeros where unused
    idx, inv = ctx.saved_tensors
    return mask_copy_cuda(g.contiguous(), inv, idx, True), None, None, None


# ------------------------------------------------------------------------------------------------
# registration: raw torch.library definitions (schema + CUDA impl + fake), which cost ~20 us per call instead of
# the ~130 us of the `torch.library.custom_op` convenience wrapper -- it matters for test-scale problems
_LIB = torch.library.Library('mrphy_b200', 'DEF')
_SCHEMAS = {'blochsim_fused_fwd': '(Tensor Mi, Tensor rf, Tensor gr, Tensor loc, Tensor? df, Tensor? b1, Tensor? T1, Tensor? T2, Tensor gamma, Tensor dt, int K, int flags, int every, int nRx=0, Tensor? rx=None) -> (Tensor, Tensor, Tensor, Tensor)', 'blochsim_fused_bwd': '(Tensor gMo, Tensor? gMt, Tensor Mo, Tensor ckpt, Tensor wave, Tensor rf, Tensor gr, Tensor loc, Tensor? df, Tensor? b1, Tensor? T1, Tensor? T2, Tensor gamma, Tensor dt, int K, int flags, int every, bool want_loc, bool want_sz, bool want_b1, Tensor? rho, Tensor? theta, Tensor? rfmax, Tensor? ts, Tensor? smax, Tensor? ddt, int rf_kind, int gr_kind, int nRx=0, Tensor? rx=None, bool want_rx=False) -> (Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor)', 'blochsim_beff_fwd': '(Tensor Mi, Tensor Beff, Tensor? T1, Tensor? T2, Tensor gamma, Tensor dt, int K, int flags) -> (Tensor, Tensor)', 'blochsim_beff_bwd': '(Tensor gMo, Tensor Mo, Tensor ckpt, Tensor Beff, Tensor? T1, Tensor? T2, Tensor gamma, Tensor dt, int K, int flags) -> (Tensor, Tensor)', 'rfgr2beff': '(Tensor rf, Tensor gr, Tensor loc, Tensor? df, Tensor? b1, Tensor gamma) -> Tensor', 'rfgr2beff_bwd': '(Tensor gB, Tensor rf, Tensor gr, Tensor loc, Tensor? b1) -> (Tensor, Tensor)', 'rfgr2beff_spin_grads': '(Tensor gB, Tensor rf, Tensor gr, bool want_loc, bool want_b1) -> (Tensor, Tensor, Tensor)', 'beff2ab': '(Tensor beff, Tensor E1, Tensor E2, Tensor gamma, Tensor dt, int K, int flags) -> (Tensor, Tensor, Tensor)', 'beff2ab_bwd': '(Tensor gA, Tensor gB, Tensor A, Tensor B, Tensor ckpt, Tensor beff, Tensor E1, Tensor E2, Tensor gamma, Tensor dt, int K, int flags) -> (Tensor, Tensor)', 'beff2uphi': '(Tensor beff, Tensor g) -> (Tensor, Tensor)', 'beff2uphi_bwd': '(Tensor? gU, Tensor? gPhi, Tensor beff, Tensor g) -> (Tensor, Tensor)', 'freeprec': '(Tensor Mi, Tensor dur, Tensor? T1, Tensor? T2, Tensor? df, bool adjoint) -> Tensor', 'design_waveform': '(Tensor? rho, Tensor? theta, Tensor? rfmax, Tensor? ts, Tensor? smax, Tensor? dt, int rf_kind, int gr_kind) -> (Tensor, Tensor)', 'design_waveform_bwd': '(Tensor? grf, Tensor? ggr, Tensor? rho, Tensor? theta, Tensor? rfmax, Tensor? ts, Tensor? smax, Tensor? dt, int rf_kind, int gr_kind) -> (Tensor, Tensor, Tensor)', 'mask_copy': '(Tensor v, Tensor idx, Tensor inv, bool fill_zero) -> Tensor', 'clamp_waveform': '(Tensor x, Tensor lim, float eps, int kind) -> Tensor', 'clamp_waveform_bwd': '(Tensor g, Tensor x, Tensor lim, float eps, int kind) -> Tensor'}


def _register(name, impl, fake):
    _LIB.define(name + _SCHEMAS[name])
    _LIB.impl(name, impl, 'CUDA')
    torch.library.register_fake('mrphy_b200::' + name, fake, lib=_LIB)
    return getattr(torch.ops.mrphy_b200, name).default


blochsim_fused_fwd = _register('blochsim_fused_fwd', _impl_blochsim_fused_fwd, _fake_blochsim_fused_fwd)
blochsim_fused_bwd = _register('blochsim_fused_bwd', _impl_blochsim_fused_bwd, _fake_blochsim_fused_bwd)
blochsim_beff_fwd = _register('blochsim_beff_fwd', _impl_blochsim_beff_fwd, _fake_blochsim_beff_fwd)
blochsim_beff_bwd = _register('blochsim_beff_bwd', _impl_blochsim_beff_bwd, _fake_blochsim_beff_bwd)
rfgr2beff_cuda = _register('rfgr2beff', _impl_rfgr2beff, _fake_rfgr2beff)
rfgr2beff_bwd_cuda = _register('rfgr2beff_bwd', _impl_rfgr2beff_bwd, _fake_rfgr2beff_bwd)
rfgr2beff_spin_grads_cuda = _register('rfgr2beff_spin_grads', _impl_rfgr2beff_spin_grads, _fake_rfgr2beff_spin_grads)
beff2ab_cuda = _register('beff2ab', _impl_beff2ab, _fake_beff2ab)
beff2ab_bwd_cuda = _register('beff2ab_bwd', _impl_beff2ab_bwd, _fake_beff2ab_bwd)
beff2uphi_cuda = _register('beff2uphi', _impl_beff2uphi, _fake_beff2uphi)
beff2uphi_bwd_cuda = _register('beff2uphi_bwd', _impl_beff2uphi_bwd, _fake_beff2uphi_bwd)
freeprec_cuda = _register('freeprec', _impl_freeprec, _fake_freeprec)
design_waveform_cuda = _register('design_waveform', _impl_design_waveform, _fake_design_waveform)
design_waveform_bwd_cuda = _register('design_waveform_bwd', _impl_design_waveform_bwd, _fake_design_waveform_bwd)
mask_copy_cuda = _register('mask_copy', _impl_mask_copy, _fake_mask_copy)
clamp_waveform_cuda = _register('clamp_waveform', _impl_clamp_waveform, lambda x, lim, eps, kind: x.new_empty(x.shape))
clamp_waveform_bwd_cuda = _register('clamp_waveform_bwd', _impl_clamp_waveform_bwd, lambda g, x, lim, eps, kind: x.new_empty(x.shape))
torch.library.register_autograd('mrphy_b200::blochsim_fused_fwd', _fused_backward, setup_context=_fused_setup, lib=_LIB)
torch.library.register_autograd('mrphy_b200::design_waveform', _design_backward, setup_context=_design_setup, lib=_LIB)
torch.library.register_autograd('mrphy_b200::mask_copy', _mask_backward, setup_context=_mask_setup, lib=_LIB)
torch.library.register_autograd('mrphy_b200::clamp_waveform', _clamp_backward, setup_context=_clamp_setup, lib=_LIB)


# ------------------------------------------------------------------------------------------------
# re-parametrisation fused into the gradient epilogue (SURVEY 8f-2).  utils.tρθ2rf / lρθ2rf / s2g / ts2g / tρθts2rfgr tag the
# waveforms they return with the design variables they came from (`tag_design`); when such a waveform reaches
# `fused_applypulse`, the simulation is recorded in autograd as a function of the DESIGN VARIABLES, and its backward evaluates
# their gradients in the tail of the simulation's own gradient epilogue -- the backward launch of the chain disappears.
# Consequence: such a waveform is no longer a node of Mo's graph.  `x.retain_grad()` / `x.register_hook()` before the call are
# honoured (two-stage path); `torch.autograd.grad(loss, [rf])` on a re-parametrised rf raises ("not used in the graph") --
# MRPHY_B200_FUSE_DESIGN=0 restores the reference's graph.
class _DesignRecord:
    __slots__ = ('tensors', 'kind', 'versions', 'out_version')

    def __init__(self, tensors, kind, out):
        self.tensors, self.kind = tensors, kind
        self.versions = tuple(t._version for t in tensors if t is not None)
        self.out_version = out._version

    def valid_for(self, out: Tensor) -> bool:      # nothing was modified in place since the chain ran
        return out._version == self.out_version and \
            self.versions == tuple(t._version for t in self.tensors if t is not None)


def tag_design(rf: Optional[Tensor], gr: Optional[Tensor], rho, theta, rfmax, ts, smax, dt, rf_kind: int, gr_kind: int):
    """Remember on rf / gr (outputs of `design_waveform_cuda`) the inputs of the chain; gr only when it IS a gradient
    (gr_kind 1: ts -> g, 2: s -> g)."""
    if rf is not None and rf_kind:
        rf._mrphy_design = _DesignRecord((rho, theta, rfmax), rf_kind, rf)
    if gr is not None and gr_kind in (1, 2):
        gr._mrphy_design = _DesignRecord((ts, smax, dt), gr_kind, gr)


def _design_of(x: Tensor, used: Tensor) -> Optional[_DesignRecord]:
    rec = getattr(x, '_mrphy_design', None)
    if rec is None or used is not x or not x.requires_grad or x.retains_grad or getattr(x, '_backward_hooks', None) \
            or not rec.valid_for(x):
        return None          # (a caller who wants dL/dx itself -- retain_grad, a hook -- gets the two-stage path)
    return rec


class _FusedDesignApply(torch.autograd.Function):
    """Mo(Mi, rf | (rho, theta), gr | ts): forward = the fused simulation on the waveforms the chain already produced;
    backward = the fused backward with the design tail."""

    @staticmethod
    def forward(ctx, Mi, rf, gr, rho, theta, ts, loc, df, b1, T1, T2, gamma, dt, rfmax, smax, ddt, K, flags, rf_kind, gr_kind):
        Mo, _, ckpt, wave = blochsim_fused_fwd(Mi, rf, gr, loc, df, b1, T1, T2, gamma, dt, K, flags, 0)
        opt = (df, b1, T1, T2, rho, theta, rfmax, ts, smax, ddt)
        ctx.has = [x is not None for x in opt]
        ctx.K, ctx.flags, ctx.kinds = K, flags, (rf_kind, gr_kind)
        ctx.save_for_backward(Mo, ckpt, wave, rf, gr, loc, gamma, dt, *[x for x in opt if x is not None])
        return Mo

    @staticmethod
    def backward(ctx, gMo):
        Mo, ckpt, wave, rf, gr, loc, gamma, dt, *rest = ctx.saved_tensors
        rest = list(rest)
        df, b1, T1, T2, rho, theta, rfmax, ts, smax, ddt = (rest.pop(0) if h else None for h in ctx.has)
        need = ctx.needs_input_grad          # Mi, rf, gr, rho, theta, ts
        rk = ctx.kinds[0] if (need[3] or need[4]) else 0
        gk = ctx.kinds[1] if need[5] else 0
        if not (need[0] or need[1] or need[2] or rk or gk):
            return (None,) * 20
        design = (rho if rk else None, theta if rk else None, rfmax if rk else None, ts if gk else None,
                  smax if gk else None, ddt if gk else None, rk, gk)
        gMi, grf, ggr, *_, grho, gtheta, gts, _ = _fused_grads(ctx, (need[0], need[1] or rk, need[2] or gk), gMo, Mo, ckpt,
                                                            wave, rf, gr, loc, df, b1, T1, T2, gamma, dt, design=design)
        return (gMi, grf if need[1] else None, ggr if need[2] else None,
                grho if (rk and need[3]) else None, gtheta if (rk and need[4]) else None, gts if gk else None) + (None,) * 14


# ------------------------------------------------------------------------------------------------
# host-side policy: checkpoint interval from the conditioning of the inverse relaxation
_ratio_cache = {}


def _collapse(x: Tensor) -> Tensor:
    """Drop stride-0 (expanded) dims so a reduction touches each stored element once."""
    for d in range(x.ndim):
        if x.shape[d] > 1 and x.stride(d) == 0:
            x = x.select(d, 0).unsqueeze(d)
    return x


def _root(t: Tensor) -> Tensor:
    """The tensor object that owns the storage a view was taken from (stable across calls for views of user data)."""
    return t._base if t._base is not None else t


_host_max = {}


def note_host_max(t: Tensor, value: float) -> None:
    """Remember max(t) for a small device tensor whose value was known on the host when it was made (a Pulse's ``dt`` built
    from a CPU scalar): `pick_ckpt_interval` then needs no device->host read for it."""
    r = _root(t)
    if len(_host_max) > 1024:
        _host_max.clear()
    _host_max[id(r)] = (weakref.ref(r), r._version, float(value))


def _cached_max(t: Tensor) -> float:
    """max(t) on the host: from `note_host_max`, else ONE device->host read, cached per tensor object and version."""
    r = _root(t)
    hit = _host_max.get(id(r))
    if hit is not None and hit[0]() is r and hit[1] == r._version and t.numel() == r.numel():
        return hit[2]
    with torch.no_grad():
        v = float(t.max().double().item())
    if t.numel() == r.numel():
        note_host_max(t, v)
    return v


def _cached_tmin(T1: Tensor, T2: Tensor) -> float:
    """min(T1, T2) on the host, one read per (T1, T2) tensor objects and in-place versions."""
    roots = (_root(T1), _root(T2))
    key = tuple(id(r) for r in roots) + tuple(tuple(x.shape) + tuple(x.stride()) + (x.storage_offset(),) for x in (T1, T2))
    hit = _ratio_cache.get(key)
    if hit is not None:
        refs, vers, v = hit
        if all(w() is r for w, r in zip(refs, roots)) and vers == tuple(r._version for r in roots):
            return v
    with torch.no_grad():
        v = float(torch.minimum(_collapse(T1).min(), _collapse(T2).min()).double().item())
    if len(_ratio_cache) > 256:
        _ratio_cache.clear()
    _ratio_cache[key] = (tuple(weakref.ref(r) for r in roots), tuple(r._version for r in roots), v)
    return v


def pick_ckpt_interval(dt: Tensor, T1: Optional[Tensor], T2: Optional[Tensor], kmax: int = K_MAX) -> int:
    """K such that exp(K*dt/min(T1,T2)) <= e^0.4, capped at `kmax` (K_MAX; K_MAX1 for the fp32 single-coil kernels).

    Needs max(dt) and min(T1, T2) on the host.  Both are cached per tensor OBJECT and in-place version (weak references
    guard against id reuse) and SEPARATELY: the spin object keeps its T1/T2 across a design loop, while every iteration
    builds a new Pulse -- whose ``dt`` normally comes from a host scalar and is registered by `note_host_max` -- so the
    loop stays free of device->host reads.  MRPHY_B200_CKPT overrides."""
    env = os.environ.get('MRPHY_B200_CKPT')
    if env:
        return max(1, min(kmax, int(env)))
    if T1 is None:
        return kmax
    tmin = _cached_tmin(T1, T2)
    r = _cached_max(dt) / tmin if tmin > 0 else float('nan')
    K = kmax if not (r > 0) else int(max(1, min(kmax, _AMPLIFY_BUDGET / r)))
    if K >= 16:
        K -= K % 16
    return K


TRIG_POLICIES = ('precise', 'mixed', 'fast', 'strict')
_policy_override = None


def set_trig_policy(name: Optional[str]) -> None:
    """Select the fp32 arithmetic policy for this process (None: back to MRPHY_B200_TRIG / the default)."""
    global _policy_override
    assert name is None or name in TRIG_POLICIES, f'policy must be one of {TRIG_POLICIES}'
    _policy_override = name


def trig_policy() -> str:
    """fp32 arithmetic policy (ignored for fp64 tensors): `set_trig_policy`, else MRPHY_B200_TRIG, else 'precise'.

    precise  (default) rotation coefficients from half-angle polynomials on the FMA pipe (|b| <= 2 pi; Cody-Waite reduction
             + Newton-refined rsqrt beyond), forward and adjoint.  Measured at full size against the fp64 oracle (B200):
             M 0.7-0.8x the reference algorithm's own fp32 error, rf/gr gradients 4e-6 (nT=1000) ... 1e-5 (nT=2000)
             relative -- the reference's own fp32 gradients: 2e-5 ... 5e-5; north_star tolerance 1e-4.
    mixed    the same forward -- M is bit-identical to 'precise' -- and MUFU.SIN/COS/RSQ in the adjoint kernel (~6 % faster):
             the MUFU bias makes the gradient error grow with nT, 4.5e-5 at nT=1000, 8.6e-5 at nT=2000: fine for short
             pulses, outside 1e-4 beyond nT ~ 2000, hence opt-in.
    fast     MUFU trigonometry everywhere: ~1.5-2x the reference's fp32 error on M, gradients 5e-5 ... 1.3e-4.
    strict   fp32 tensors in and out, fp64 arithmetic inside (the fp64 kernels): M within 1e-5 -- in fact 3e-8 -- of the
             reference's fp64 result at every nT, which no fp32 evaluation of this recurrence, the reference's own included,
             achieves beyond nT ~ 500; costs ~2.7x the time."""
    pol = _policy_override or os.environ.get('MRPHY_B200_TRIG', 'precise')
    if pol not in TRIG_POLICIES:
        raise ValueError(f'MRPHY_B200_TRIG={pol!r}: expected one of {TRIG_POLICIES}')
    return pol


def default_flags() -> int:
    """C-ABI flags of the current `trig_policy` ('strict' is handled above the ABI: it runs the fp64 kernels)."""
    pol = trig_policy()
    if pol == 'mixed':
        return _cabi.FLAG_TRIG_PRECISE | _cabi.FLAG_TRIG_FAST_BWD
    return 0 if pol == 'fast' else _cabi.FLAG_TRIG_PRECISE


def fused_applypulse(M_: Tensor, rf: Tensor, gr: Tensor, loc_: Tensor, *, Δf_: Optional[Tensor] = None,
                     b1Map_: Optional[Tensor] = None, T1_: Optional[Tensor] = None, T2_: Optional[Tensor] = None,
                     γ_: Tensor, dt: Tensor, ckpt: Optional[int] = None, flags: Optional[int] = None,
                     record: Optional[int] = None, readout: Optional[int] = None, rxMap_: Optional[Tensor] = None):
    """Fused waveform -> magnetisation op on compact arrays; differentiable wrt ``M_``, ``rf``, ``gr`` and the spins'
    ``loc_``, ``Δf_``, ``b1Map_``, ``γ_`` (as the reference's autograd through rfgr2beff; γ only through ``Δf_/γ``).

    ``M_`` (N,nM,3), ``rf`` (N,2,nT[,nCoils]), ``gr`` (N,3,nT), ``loc_`` (N,nM,3), ``Δf_`` (N,nM),
    ``b1Map_`` (N,nM,2[,nCoils]), ``T1_/T2_/γ_`` broadcastable to (N,nM), ``dt`` () or (N|1,).

    The per-spin gradients are sums over time that the fused backward forms per spin, without the dense field.  When one
    of those inputs requires grad, a re-parametrised rf / gr (``tag_design``) is differentiated in two stages -- the
    simulation's backward, then the chain's own adjoint -- as with ``MRPHY_B200_FUSE_DESIGN=0``.

    ``record = s`` (an integer, 1 <= s <= nT) also returns the magnetisation during the pulse: ``(M, Mt)`` instead of ``M``,
    ``Mt`` (N,nM,nR,3) with nR = nT // s and ``Mt[:, :, r]`` the state after (r+1)·s steps in the lab frame -- what ``M``
    is for the pulse cut to its first (r+1)·s samples (the last entry is ``M`` when s divides nT).  ``Mt`` is a permuted
    view of the kernel's (N,nR,xyz,nM) output and is not contiguous.  Losses on ``Mt``, on ``M`` or on both are
    differentiable like ``M`` alone; a re-parametrised waveform is then differentiated in two stages, as above.

    ``readout = s`` (an integer, 1 <= s <= nT) returns ``(M, S)``, the receive signal of the same states summed over the spins
    inside the kernels: ``S[n, 0, r] + i S[n, 1, r] = sum_i (cx + i cy)[n, i] (Mx + i My)[n, i]`` after (r+1)·s steps, with
    the receive map ``rxMap_`` (N,nM,xy[,nRx]) (1 <= nRx <= 16; None: c = 1).  No conjugation and no scale factor.  ``S`` is
    (N,2,nR), or (N,2,nR,nRx) when ``rxMap_`` has the coil dimension; it is bitwise reproducible run to run.  Losses on ``S``,
    ``M`` or both reach everything ``M`` reaches and ``rxMap_``.  Not together with ``record``.
    """
    if record is not None:
        record = _check_record(record, rf, b1Map_)
    if readout is not None:
        readout = _check_readout(readout, record, rf, b1Map_, rxMap_)
    _require_cuda(M_, rf, gr, loc_, Δf_, b1Map_, T1_, T2_)
    dtype, dev = M_.dtype, M_.device
    if dtype not in _F:
        raise TypeError(f'mrphy (B200): M must be float32 or float64, got {dtype}')
    if dtype == torch.float32 and flags is None and trig_policy() == 'strict':
        # fp32 tensors in and out, fp64 arithmetic: the casts are differentiable torch copies either side of the fp64 op.
        # The checkpoint interval is taken from the caller's own tensors (cached per object: no host read per call, which
        # the fresh fp64 copies would force -- and which would invalidate a CUDA-graph capture).
        mv = lambda x: None if x is None else (on_device(x, dev) if x.dtype in _F else on_device(x, dev, dtype))
        K = int(ckpt) if ckpt is not None else pick_ckpt_interval(mv(dt), mv(T1_), mv(T2_))
        up = lambda x: None if x is None else x.to(torch.float64)
        out = fused_applypulse(up(M_), up(rf), up(gr), up(loc_), Δf_=up(Δf_), b1Map_=up(b1Map_), T1_=up(T1_), T2_=up(T2_),
                               γ_=γ_, dt=dt, ckpt=K, record=record, readout=readout, rxMap_=up(rxMap_))
        if record is not None or readout is not None:
            return out[0].to(torch.float32), out[1].to(torch.float32)
        return out.to(torch.float32)
    assert (T1_ is None) == (T2_ is None)      # both or neither (sims.py:68)
    N, nM = loc_.shape[0], loc_.shape[1]
    assert M_.shape == (N, nM, 3) and loc_.shape == (N, nM, 3)
    assert rf.shape[0] == N and rf.shape[1] == 2 and gr.shape == (N, 3, rf.shape[2])
    cast = lambda x: None if x is None else x.to(device=dev, dtype=dtype)
    move = lambda x: None if x is None else (on_device(x, dev) if x.dtype in _F else on_device(x, dev, dtype))
    rf_in, gr_in = rf, gr
    rf, gr = cast(rf), cast(gr)
    Mi = _inner_contig(cast(M_), 1)
    loc = _inner_contig(cast(loc_), 1)
    b1 = cast(b1Map_)
    if b1 is not None:
        if b1.ndim == 3:
            b1 = b1[..., None]
        nC = rf.shape[3] if rf.ndim == 4 else 1
        if nC == 1 and b1.shape[3] > 1:          # one rf for every coil: sum_c b1_c * rf = (sum_c b1_c) * rf
            b1 = b1.sum(dim=3, keepdim=True)
        assert b1.shape[2] == 2 and b1.shape[3] in (1, nC), 'b1Map and rf disagree on nCoils'
        # a single-coil b1Map with multi-coil rf broadcasts over coils, as upstream (beffective.py:153-165)
        b1 = _inner_contig(b1.expand(N, nM, 2, nC) if tuple(b1.shape) != (N, nM, 2, nC) else b1, 2)
    df, T1, T2, gam, dtt = (move(x) for x in (Δf_, T1_, T2_, γ_, dt))
    one_channel = b1 is None or b1.shape[3] == 1
    K = int(ckpt) if ckpt is not None else pick_ckpt_interval(dtt, T1, T2, K_MAX1 if (dtype == torch.float32 and one_channel) else K_MAX)
    if ckpt is None and dtype == torch.float32 and b1 is not None and b1.shape[3] >= 3:
        K = min(K, TC_K_MAX)                     # the tensor-core kernels stage 32 steps per chunk
    fl = default_flags() if flags is None else flags
    spin_grad = any(x is not None and x.requires_grad for x in (loc_, Δf_, b1Map_, γ_))
    if torch.is_grad_enabled() and not spin_grad and record is None and readout is None and \
            os.environ.get('MRPHY_B200_FUSE_DESIGN', '1') != '0':
        # rf and/or gr straight out of the re-parametrisation chain: differentiate w.r.t. the design variables in the
        # simulation's own gradient epilogue (see _FusedDesignApply)
        r_rf, r_gr = _design_of(rf_in, rf), _design_of(gr_in, gr)
        if r_rf is not None or r_gr is not None:
            rho, theta, rfmax = r_rf.tensors if r_rf is not None else (None, None, None)
            ts, smax, ddt = r_gr.tensors if r_gr is not None else (None, None, None)
            return _FusedDesignApply.apply(Mi, rf.detach() if r_rf is not None else rf, gr.detach() if r_gr is not None else gr,
                                           rho, theta, ts, loc, df, b1, T1, T2, gam, dtt, rfmax, smax, ddt, K, fl,
                                           r_rf.kind if r_rf is not None else 0, r_gr.kind if r_gr is not None else 0)
    if readout is not None:
        rx, coil_dim = cast(rxMap_), rxMap_ is not None and rxMap_.ndim == 4
        if rx is not None:
            rx = rx if coil_dim else rx[..., None]
            assert rx.ndim == 4 and rx.shape[0] in (1, N) and rx.shape[1] in (1, nM) and rx.shape[2] == 2, \
                f'rxMap_ of shape {tuple(rxMap_.shape)} is not (N|1, nM|1, 2[, nRx])'
            rx = _inner_contig(rx.expand(N, nM, 2, rx.shape[3]), 2)   # broadcasts stay stride 0: no copy
        Mo, S, _, _ = blochsim_fused_fwd(Mi, rf, gr, loc, df, b1, T1, T2, gam, dtt, K, fl, readout,
                                         1 if rx is None else rx.shape[3], rx)
        return Mo, (S if coil_dim else S[..., 0])
    Mo, Mt, _, _ = blochsim_fused_fwd(Mi, rf, gr, loc, df, b1, T1, T2, gam, dtt, K, fl, record or 0)
    return Mo if record is None else (Mo, Mt.permute(0, 3, 1, 2))


def _check_record(record, rf: Tensor, b1Map_: Optional[Tensor]) -> int:
    """The record stride `fused_applypulse` takes, or ValueError (before anything runs)."""
    if isinstance(record, bool) or not isinstance(record, numbers.Integral):
        raise ValueError(f'mrphy (B200): record must be an integer number of steps, got {record!r}')
    nT = rf.shape[2]
    if not 1 <= record <= nT:
        raise ValueError(f'mrphy (B200): record={record} is outside [1, nT = {nT}]')
    if b1Map_ is not None and rf.ndim == 4 and rf.shape[3] > 16:
        raise ValueError(f'mrphy (B200): record needs the fused kernels, which take at most 16 transmit coils with a b1Map '
                         f'(got {rf.shape[3]}); the explicit-Beff route does not record')
    return int(record)


def _check_readout(readout, record, rf: Tensor, b1Map_: Optional[Tensor], rxMap_: Optional[Tensor]) -> int:
    """The readout stride `fused_applypulse` takes, or ValueError (before anything runs)."""
    if isinstance(readout, bool) or not isinstance(readout, numbers.Integral):
        raise ValueError(f'mrphy (B200): readout must be an integer number of steps, got {readout!r}')
    nT = rf.shape[2]
    if not 1 <= readout <= nT:
        raise ValueError(f'mrphy (B200): readout={readout} is outside [1, nT = {nT}]')
    if record is not None:
        raise ValueError('mrphy (B200): readout and record do not combine in one call')
    if rxMap_ is not None and rxMap_.ndim == 4 and rxMap_.shape[3] > 16:
        raise ValueError(f'mrphy (B200): readout takes at most 16 receive coils (got {rxMap_.shape[3]})')
    if b1Map_ is not None and rf.ndim == 4 and rf.shape[3] > 16:
        raise ValueError(f'mrphy (B200): readout needs the fused kernels, which take at most 16 transmit coils with a b1Map '
                         f'(got {rf.shape[3]}); the explicit-Beff route has no readout')
    return int(readout)
