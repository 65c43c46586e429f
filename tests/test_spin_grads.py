"""Per-spin gradients (loc, Δf, b1Map, γ) from the fused backward, against the fp64 oracle, the explicit-field route and
finite differences; the C-ABI mirror and the fake of the new op need no GPU."""
import ctypes
import re

import pytest
import torch
from torch import tensor

f32, f64 = torch.float32, torch.float64


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available(), 'run with -m gpu on a CUDA box'
    from mrphy import _cabi
    _cabi.lib()
    return torch.device('cuda:0')


def rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def _problem(seed, N, nM, nT, nC, has_b1=True, relax=True, zero_b1=0):
    """Seeded fp64 inputs: per-batch dt, per-spin γ; nC = 0: rf without a coil dimension.  The first `zero_b1` spins of
    every batch entry have b1 = 0 (identity frame of the single-coil kernels)."""
    gen = torch.Generator().manual_seed(seed)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    p = dict(rf=U(N, 2, nT, nC) * 0.1 if nC else U(N, 2, nT) * 0.1, gr=U(N, 3, nT) * 2, loc=U(N, nM, 3) * 12,
             df=U(N, nM) * 200, b1=None, M0=torch.nn.functional.normalize(U(N, nM, 3), dim=-1),
             gam=4257.6 * (1 + 0.02 * U(N, nM)), dt=4e-6 * (1 + 0.25 * U(N).abs()),
             T1=(1.0 + 0.5 * U(N, nM)) if relax else None, T2=(0.06 + 0.05 * U(N, nM)) if relax else None, w=U(N, nM, 3))
    if has_b1:
        b1 = U(N, nM, 2, max(nC, 1)) * 0.3
        b1[:, :, 0] += 1
        b1[:, :zero_b1] = 0
        p['b1'] = b1
    return p


def _beff(rf, gr, loc, df, b1, gam):
    """oracle.bloch_oracle.rfgr2beff (beffective.py:107-168) written on tensors that keep their autograd graph."""
    N, nM = loc.shape[0], loc.shape[1]
    bz = torch.einsum('nmc,nct->nmt', loc, gr)
    if df is not None:
        bz = bz + (df / gam)[..., None]
    rf = rf if rf.ndim == 4 else rf[..., None]
    rx, ry = rf[:, 0], rf[:, 1]
    if b1 is None:
        bx, by = rx.sum(-1)[:, None].expand(N, nM, -1), ry.sum(-1)[:, None].expand(N, nM, -1)
    else:
        br, bi = b1[:, :, 0], b1[:, :, 1]
        bx = torch.einsum('nmc,ntc->nmt', br, rx) - torch.einsum('nmc,ntc->nmt', bi, ry)
        by = torch.einsum('nmc,ntc->nmt', br, ry) + torch.einsum('nmc,ntc->nmt', bi, rx)
    return torch.stack([bx, by, bz], dim=-1)


SPIN = ('loc', 'df', 'b1', 'gam')                         # the per-spin inputs that can require grad
PER_SPIN = ('M0', 'loc', 'df', 'b1', 'gam', 'T1', 'T2', 'w')  # problem entries with a spin axis (dim 1)
_ORACLE = {}                                               # (problem content, dtype) -> oracle result, solved once


def _subset(p, sub):
    return p if sub is None else {k: (v[:, sub] if k in PER_SPIN and v is not None else v) for k, v in p.items()}


def _fingerprint(p):
    import hashlib
    return tuple((k, None) if v is None else (k, tuple(v.shape), str(v.dtype),
                                              hashlib.sha1(v.detach().contiguous().numpy().tobytes()).hexdigest())
                 for k, v in sorted(p.items()))


def _solve(p, dtype):
    from oracle import bloch_oracle as orc
    p = {k: (None if v is None else (v if k in ('gam', 'dt') else v.to(dtype))) for k, v in p.items()}
    leaves = {k: p[k].to(dtype).clone().requires_grad_(True) for k in SPIN + ('rf', 'gr') if p[k] is not None}
    q = dict(p, **leaves)
    B = _beff(q['rf'], q['gr'], q['loc'], q['df'], q['b1'], q['gam'])
    assert torch.allclose(B.detach(), orc.rfgr2beff(p['rf'], p['gr'], p['loc'], p['df'], p['b1'], gamma=p['gam'], dtype=dtype),
                          atol=1e-12 if dtype == f64 else 1e-4)
    Mo, gM0, gB = orc.blochsim_adj(p['M0'], B.detach(), p['w'], p['T1'], p['T2'], gamma=p['gam'], dt=p['dt'], dtype=dtype)
    (B * gB).sum().backward()
    return Mo.double(), dict({k: v.grad.double() for k, v in leaves.items() if v.grad is not None}, M0=gM0.double())


def _oracle(p, dtype=f64, sub=None, full=False):
    """dL/d(loc, Δf, b1Map, γ) and Mo of L = sum(w * Mo): dL/dBeff from the oracle's adjoint, then autograd of the field.

    `dtype` is the arithmetic of the reference algorithm (fp32: its own rounding, the floor of the fp32 checks); `sub`
    restricts the problem to those spins first -- spins are independent, so every per-spin result of a subset is that of
    the whole problem.  `full` adds dL/dM0, dL/drf and dL/dgr (the latter two are sums over the spins solved).  Each
    (problem, dtype, subset) is solved once per module."""
    q = _subset(p, sub)
    key = (_fingerprint(q), dtype)
    if key not in _ORACLE:
        _ORACLE[key] = _solve(q, dtype)
    Mo, g = _ORACLE[key]
    return Mo, {k: v for k, v in g.items() if full or k in SPIN}


def _as32(p):
    """The inputs an fp32 run is handed (γ and dt stay fp64 constants), in fp64."""
    return {k: (None if v is None else (v if k in ('gam', 'dt') else v.float().double())) for k, v in p.items()}


def _refs(p, dtype, sub=None):
    """-> (fp64 reference, the reference algorithm in fp32 on the same inputs, or None for fp64), both with full=True."""
    if dtype == f64:
        return _oracle(p, f64, sub, True), None
    q = _as32(p)
    return _oracle(q, f64, sub, True), _oracle(q, f32, sub, True)


def _fused(p, dev, dtype, K=None, flags=None, rf_grad=True, gr_grad=None, spin=SPIN, m0_grad=False, policy=None, sub=None):
    """fused_applypulse with the spin inputs `spin`, rf (`rf_grad`), gr (`gr_grad`, default: as rf) and M0 (`m0_grad`)
    requiring grad, under the fp32 `policy` -> (Mo, {'M0', 'loc', 'df', 'b1', 'gam', 'rf', 'gr': .grad or None}).
    `sub`: Mo and the per-spin gradients of those spins only."""
    from mrphy import _ops
    gr_grad = rf_grad if gr_grad is None else gr_grad
    kw = {'dtype': dtype, 'device': dev}
    t = {k: (None if v is None else v.to(**kw)) for k, v in p.items()}
    t['gam'], t['dt'] = p['gam'].to(dev), p['dt'].to(dev)             # fp64 constants next to fp32 state
    leaves = [k for k in spin if t[k] is not None] + [k for k, on in (('rf', rf_grad), ('gr', gr_grad), ('M0', m0_grad)) if on]
    for k in leaves:
        t[k].requires_grad_(True)
    _ops.set_trig_policy(policy)
    try:
        Mo = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'],
                                   T2_=t['T2'], γ_=t['gam'], dt=t['dt'], ckpt=K, flags=flags)
        (Mo * t['w']).sum().backward()
    finally:
        _ops.set_trig_policy(None)
    g = {k: (None if t[k] is None else t[k].grad) for k in ('M0',) + SPIN + ('rf', 'gr')}
    if sub is not None:
        g = {k: (v[:, sub] if k in PER_SPIN and v is not None else v) for k, v in g.items()}
        Mo = Mo[:, sub]
    return Mo.detach(), g


def _check(p, dev, dtype, tol, K=None):
    Mo_ref, ref = _oracle(p)
    Mo, g = _fused(p, dev, dtype, K)
    for k, v in ref.items():
        assert g[k] is not None and g[k].shape == p[k].shape, k
        assert rel(g[k], v) < tol, (k, rel(g[k], v))


@pytest.mark.gpu
@pytest.mark.parametrize('dtype,tol', [(f64, 1e-9), (f32, 1e-4)])
@pytest.mark.parametrize('case', ['one_coil_zero_b1', 'no_b1', 'nC2', 'nC3', 'nC4', 'nC8', 'nC16', 'no_relax', 'rf_no_coil_dim'])
def test_against_oracle(dev, dtype, tol, case):
    N, nM, nT = 2, 261, 97
    kw = dict(one_coil_zero_b1=dict(nC=1, zero_b1=5), no_b1=dict(nC=1, has_b1=False), nC2=dict(nC=2), nC3=dict(nC=3),
              nC4=dict(nC=4), nC8=dict(nC=8), nC16=dict(nC=16), no_relax=dict(nC=1, relax=False),
              rf_no_coil_dim=dict(nC=0))[case]
    _check(_problem(100 + len(case) * 7 + kw['nC'], N, nM, nT, **kw), dev, dtype, tol)


@pytest.mark.gpu
@pytest.mark.parametrize('K,nC', [(1, 1), (7, 1), (64, 1), (128, 1), (1, 4), (7, 2), (64, 8)])   # 128: fp32 single coil only
def test_checkpoint_intervals(dev, K, nC):
    p = _problem(40 + K + nC, 1, 200, 301, nC)                        # nT not a multiple of K
    _check(p, dev, f64, 1e-9, min(K, 64))
    _check(p, dev, f32, 1e-4, K)


@pytest.mark.gpu
@pytest.mark.parametrize('trig,nT', [('precise', 203), ('mixed', 203), ('fast', 203), ('strict', 203), ('precise', 2000),
                                     ('strict', 2000)])
def test_fp32_policies(dev, trig, nT):
    from mrphy import _ops
    p = _problem(7, 1, 333, nT, 1)
    _ops.set_trig_policy(trig)
    try:
        _check(p, dev, f32, 1e-4)
    finally:
        _ops.set_trig_policy(None)


@pytest.mark.gpu
@pytest.mark.parametrize('nC', [1, 8])
def test_against_explicit_route_and_fd(dev, nC):
    """The explicit composition sims.blochsim(M, pulse2beff(...)) on the same inputs; fp64 central finite differences."""
    from mrphy import mobjs, sims
    p = _problem(3 + nC, 1, 150, 60, nC, zero_b1=2)
    for dtype, tol in ((f64, 1e-9), (f32, 1e-4)):
        kw = {'dtype': dtype, 'device': dev}
        sp = mobjs.SpinArray((1, 150), **kw)
        pulse = mobjs.Pulse(rf=p['rf'].to(**kw), gr=p['gr'].to(**kw), dt=tensor(4e-6, dtype=f64), **kw)
        w = p['w'].to(**kw)
        grads = []
        for explicit in (False, True):
            loc, df, b1 = (p[k].to(**kw).requires_grad_(True) for k in ('loc', 'df', 'b1'))
            if explicit:
                M = sims.blochsim(sp.M_, sp.pulse2beff(pulse, loc_=loc, Δf_=df, b1Map_=b1), T1=sp.T1_, T2=sp.T2_, γ=sp.γ_,
                                  dt=pulse.dt)
            else:
                M = sp.applypulse(pulse, loc_=loc, Δf_=df, b1Map_=b1)
            (M * w).sum().backward()
            grads.append((loc.grad, df.grad, b1.grad))
        for a, b in zip(*grads):
            assert rel(a, b) < tol
        if dtype == f64:
            f = lambda l, d, b: float((sp.applypulse(pulse, loc_=l, Δf_=d, b1Map_=b) * w).sum())
            base = [p[k].to(**kw) for k in ('loc', 'df', 'b1')]
            for which, idx in ((0, (0, 3, 2)), (1, (0, 7)), (2, (0, 1, 0, 0)), (2, (0, 4, 1, nC - 1))):
                eps = 1e-6
                hi, lo = [x.clone() for x in base], [x.clone() for x in base]
                hi[which][idx] += eps
                lo[which][idx] -= eps
                fd = (f(*hi) - f(*lo)) / (2 * eps)
                assert abs(fd - float(grads[0][which][idx])) < 1e-6 * max(1.0, abs(fd))


@pytest.mark.gpu
@pytest.mark.parametrize('tag', ['b1bc', 'rfbc'])
def test_broadcast_coils_against_explicit_route(dev, tag):
    """tests/golden/standalone.npz's coil broadcasts: a one-coil b1Map driving multi-coil rf (b1bc), a multi-coil b1Map with
    one rf for every coil (rfbc); gradients reach b1Map in its own shape."""
    import os
    import numpy as np
    from mrphy import mobjs, sims
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'standalone.npz'))
    kw = {'dtype': f64, 'device': dev}
    rf, gr, loc, b1 = (torch.as_tensor(g[f'b_{tag}_{k}']).to(**kw) for k in ('rf', 'gr', 'loc', 'b1'))
    N, nM = loc.shape[0], loc.shape[1]
    sp = mobjs.SpinArray((N, nM), **kw)
    pulse = mobjs.Pulse(rf=rf, gr=gr, **kw)
    df0 = torch.linspace(-50, 50, N * nM, **kw).reshape(N, nM)
    grads = []
    for explicit in (False, True):
        l, b, d = loc.clone().requires_grad_(True), b1.clone().requires_grad_(True), df0.clone().requires_grad_(True)
        M = sims.blochsim(sp.M_, sp.pulse2beff(pulse, loc_=l, Δf_=d, b1Map_=b), T1=sp.T1_, T2=sp.T2_, γ=sp.γ_,
                          dt=pulse.dt) if explicit else sp.applypulse(pulse, loc_=l, Δf_=d, b1Map_=b)
        (M * M.detach()).sum().backward()
        grads.append((l.grad, b.grad, d.grad))
    for a, b in zip(*grads):
        assert a.shape == b.shape and rel(a, b) < 1e-9


@pytest.mark.gpu
def test_nothing_else_moves_and_reproducible(dev):
    """Mo, rf.grad, gr.grad, M_.grad bitwise as without per-spin gradients; per-spin gradients bitwise run to run."""
    from mrphy import _ops
    for nC, dtype in ((1, f32), (2, f32), (8, f32), (1, f64), (4, f64)):
        p = _problem(11, 1, 4000, 300, nC)
        kw = {'dtype': dtype, 'device': dev}
        out = []
        for spin in (False, True, True):
            t = {k: (None if v is None else v.to(**kw)) for k, v in p.items()}
            for k in ('rf', 'gr', 'M0') + (('df', 'b1', 'loc') if spin else ()):
                t[k].requires_grad_(True)
            Mo = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'],
                                       T2_=t['T2'], γ_=t['gam'], dt=t['dt'])
            (Mo * t['w']).sum().backward()
            out.append([Mo.detach(), t['rf'].grad, t['gr'].grad, t['M0'].grad] +
                       ([t['df'].grad, t['b1'].grad, t['loc'].grad] if spin else []))
        for a, b in zip(out[0], out[1]):
            assert torch.equal(a, b)
        for a, b in zip(out[1], out[2]):
            assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize('nC', [1, 8])
def test_fixed_pulse_skips_finalize(dev, nC):
    """Only Δf_ / b1Map_ requiring grad: the backward issues one launch fewer (no gradient finalize) and still agrees."""
    from mrphy import _cabi
    p = _problem(5, 1, 500, 120, nC)
    counts = []
    for rf_grad in (True, False):
        before = _cabi.launch_counter
        _fused(p, dev, f64, rf_grad=rf_grad)
        counts.append(_cabi.launch_counter - before)
    assert counts[1] == counts[0] - 1, counts
    _, ref = _oracle(p)
    _, g = _fused(p, dev, f64, rf_grad=False)
    for k in ('df', 'b1', 'loc', 'gam'):
        assert rel(g[k], ref[k]) < 1e-9


@pytest.mark.gpu
def test_public_api_masked_cube_and_sequence(dev):
    from mrphy import mobjs, sims
    kw = {'dtype': f64, 'device': dev}
    n = 8
    ax = torch.arange(n) - n // 2
    mask = ((ax[:, None, None] ** 2 + ax[None, :, None] ** 2 + ax[None, None, :] ** 2) < (n // 2) ** 2)[None].to(dev)
    gen = torch.Generator().manual_seed(2)
    U = lambda *s: (torch.rand(s, generator=gen, dtype=f64) * 2 - 1).to(dev)
    cube = mobjs.SpinCube((1, n, n, n), tensor([[24., 24., 24.]]), mask=mask, **kw)
    df = (U(1, n, n, n) * 100).requires_grad_(True)
    b1 = (U(1, n, n, n, 2) * 0.2 + tensor([1., 0.], **kw)).requires_grad_(True)
    cube.Δf = df
    pulse = mobjs.Pulse(rf=U(1, 2, 50) * 0.1, gr=U(1, 3, 50) * 2, **kw)
    M = cube.applypulse(pulse, b1Map=b1, doEmbed=True)
    M_ = cube.extract(M)
    (M_ * M_.detach()).sum().backward()
    outside = ~mask[0]
    assert df.grad is not None and b1.grad is not None
    assert float(df.grad[0][outside].abs().max()) == 0 and float(b1.grad[0][outside].abs().max()) == 0
    assert float(df.grad[0][mask[0]].abs().max()) > 0 and float(b1.grad[0][mask[0]].abs().max()) > 0
    # the compact values: the oracle on the masked spins alone
    c = lambda x: x.detach().cpu().double()
    w = c(M_)
    q = dict(rf=c(pulse.rf), gr=c(pulse.gr), loc=c(cube.loc_), df=c(cube.extract(df)), b1=c(cube.extract(b1))[..., None],
             M0=c(cube.M_), gam=c(cube.γ_), dt=c(pulse.dt), T1=c(cube.T1_), T2=c(cube.T2_), w=w)
    _, ref = _oracle(q)
    _agree('df', cube.extract(df.grad), ref['df'])
    _agree('b1', cube.extract(b1.grad), ref['b1'][..., 0])
    # a sequence with a gap: the same Δf_, loc_ and b1Map_ gradients as the explicit route (freeprec adds none to the
    # latter two, and its own to Δf_, as upstream)
    sp = mobjs.SpinArray((1, 64), **kw)
    loc, dfl = U(1, 64, 3) * 5, U(1, 64) * 100
    b1l = U(1, 64, 2) * 0.2 + tensor([1., 0.], **kw)
    gap = tensor(1e-3, dtype=f64)
    grads = []
    for explicit in (False, True):
        d, l, b = dfl.clone().requires_grad_(True), loc.clone().requires_grad_(True), b1l.clone().requires_grad_(True)
        if explicit:
            M = sp.M_
            for ev in (pulse, gap, pulse):
                M = sims.freeprec(M, gap.to(dev), T1=sp.T1_, T2=sp.T2_, Δf=d) if ev is gap else \
                    sims.blochsim(M, sp.pulse2beff(ev, loc_=l, Δf_=d, b1Map_=b), T1=sp.T1_, T2=sp.T2_, γ=sp.γ_, dt=ev.dt)
        else:
            M = sp.applysequence([pulse, gap, pulse], loc_=l, Δf_=d, b1Map_=b)
        M.sum().backward()
        grads.append((d.grad, l.grad, b.grad))
    for name, a, b in zip(('df', 'loc', 'b1'), *grads):
        _agree(name, a, b)


@pytest.mark.gpu
def test_scale_memory(dev):
    """128³ spins x 2000 steps, fp32: Δf_ and b1Map_ gradients cost at most 1.1x the memory of the rf/gr-only step + 256 MB
    (the dense field and its gradient would need ~100 GB), and agree with the oracle on 256 seeded spins."""
    from mrphy import _ops
    nM, nT = 128 ** 3, 2000
    gen = torch.Generator(device=dev).manual_seed(0)
    U = lambda *s: torch.rand(s, generator=gen, device=dev) * 2 - 1
    M0 = torch.nn.functional.normalize(U(1, nM, 3), dim=-1)
    loc, df0 = U(1, nM, 3) * 12, U(1, nM) * 100
    b10 = U(1, nM, 2) * 0.1 + tensor([1., 0.], device=dev)
    rf, gr = (U(1, 2, nT) * 0.1).requires_grad_(True), (U(1, 3, nT) * 2).requires_grad_(True)
    peaks = []
    for spin in (False, True):
        df, b1 = df0.clone().requires_grad_(spin), b10.clone().requires_grad_(spin)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        Mo = _ops.fused_applypulse(M0, rf, gr, loc, Δf_=df, b1Map_=b1, γ_=tensor(4257.6, dtype=f64), dt=tensor(4e-6, dtype=f64))
        Mo.sum().backward()
        torch.cuda.synchronize()
        peaks.append(torch.cuda.max_memory_allocated() - base)
        del Mo
        rf.grad = gr.grad = None
    assert peaks[1] <= 1.1 * peaks[0] + 256 * 2 ** 20, peaks
    sub = torch.randperm(nM, generator=torch.Generator().manual_seed(3))[:256].to(dev)
    c = lambda x: x.detach()[:, sub].cpu().double()
    q = dict(rf=rf.detach().cpu().double(), gr=gr.detach().cpu().double(), loc=c(loc), df=c(df0), b1=c(b10)[..., None],
             M0=c(M0), gam=torch.full((1, 256), 4257.6, dtype=f64), dt=tensor(4e-6, dtype=f64), T1=None, T2=None,
             w=torch.ones(1, 256, 3, dtype=f64))
    (_, ref), r32 = _refs(q, f32)
    _agree('df', df.grad[:, sub], ref['df'], r32[1]['df'])
    _agree('b1', b1.grad[:, sub], ref['b1'][..., 0], r32[1]['b1'][..., 0])


@pytest.mark.gpu
def test_graph_capture(dev):
    from mrphy import graphs, mobjs
    kw = {'dtype': f32, 'device': dev}
    gen = torch.Generator().manual_seed(4)
    U = lambda *s: (torch.rand(s, generator=gen) * 2 - 1).to(dev)
    sp = mobjs.SpinArray((1, 2000), **kw)
    loc = U(1, 2000, 3) * 5
    df = (U(1, 2000) * 100).requires_grad_(True)
    b1 = (U(1, 2000, 2) * 0.1 + tensor([1., 0.], **kw)).requires_grad_(True)
    pulse = mobjs.Pulse(rf=(U(1, 2, 100) * 0.1).requires_grad_(True), gr=(U(1, 3, 100) * 2).requires_grad_(True), **kw)
    step = graphs.capture(lambda: sp.applypulse(pulse, loc_=loc, Δf_=df, b1Map_=b1).sum().backward(),
                          params=[df, b1, pulse.rf, pulse.gr])
    step.replay()
    first = [df.grad.clone(), b1.grad.clone(), pulse.rf.grad.clone()]
    step.replay()
    torch.cuda.synchronize()
    for a, b in zip(first, (df.grad, b1.grad, pulse.rf.grad)):
        assert torch.equal(a, b)
    d2, b2 = df.detach().clone().requires_grad_(True), b1.detach().clone().requires_grad_(True)
    sp.applypulse(pulse, loc_=loc, Δf_=d2, b1Map_=b2).sum().backward()
    assert rel(first[0], d2.grad) < 1e-6 and rel(first[1], b2.grad) < 1e-6


@pytest.mark.gpu
def test_more_than_16_coils_keeps_explicit_route(dev):
    """More than 16 transmit coils with a b1Map, loc requiring grad: the fused kernels refuse these inputs, so applypulse
    keeps the explicit route -- the same field and magnetisation as the explicit composition, and the same refusal of
    the backward, whose per-spin pass over dL/dBeff (rfgr2beff_spin_grads) takes at most 16 coils."""
    from mrphy import mobjs, sims
    kw = {'dtype': f64, 'device': dev}
    p = _problem(17, 1, 40, 30, 20)
    sp = mobjs.SpinArray((1, 40), **kw)
    pulse = mobjs.Pulse(rf=p['rf'].to(**kw), gr=p['gr'].to(**kw), **kw)
    b1 = p['b1'].to(**kw)
    out, errors = [], []
    for explicit in (False, True):
        loc = p['loc'].to(**kw).requires_grad_(True)
        M = sims.blochsim(sp.M_, sp.pulse2beff(pulse, loc_=loc, b1Map_=b1), T1=sp.T1_, T2=sp.T2_, γ=sp.γ_,
                          dt=pulse.dt) if explicit else sp.applypulse(pulse, loc_=loc, b1Map_=b1)
        out.append(M.detach())
        with pytest.raises(RuntimeError, match='more than 16 transmit coils') as e:
            M.sum().backward()
        errors.append(str(e.value))
    assert torch.equal(out[0], out[1])
    assert errors[0] == errors[1]


# ---- every SG kernel, multi-tile CTAs, broadcasts, routes: per-spin checks ----------------------------------------------
# fp32 per-spin bound: max(1e-4, c x the reference algorithm's own fp32 e_s on the same spin).  Measured on a B200 (1000 W)
# over every fp32 case below: with 'precise' no spin of any output exceeds 1e-4 (largest e_s 1.5e-5; 'strict' 5.8e-8), so
# c = 2 never binds there.  With MUFU trigonometry ('fast'; 'mixed' in the adjoint) one spin of dL/db1Map
# (2 coils, no relaxation, packed and generic kernel alike) reaches e_s = 1.3e-4, 137x the reference's own fp32 error on
# that spin, while 'precise' on the same problem stays at 5.3e-6: the documented error of the MUFU policies (see
# mrphy._ops.trig_policy), not of the spin-gradient fold -- hence c = 200 for those two policies only.
C32 = 2.0
C32_MUFU = 200.0


def _spins(x):
    """(spins, components): the leading (N, nM) axes are the spins; a tensor without them is one row per entry / one row."""
    x = x.detach().cpu().double()
    return x.reshape(x.shape[0] * x.shape[1], -1) if x.ndim >= 2 else x.reshape(-1, 1) if x.ndim == 1 else x.reshape(1, 1)


def _es(g, r):
    """e_s = |g_s - r_s| / max(|r_s|, rms_s |r_s|) per spin: one norm over the whole tensor hides a few wrong spins."""
    g, r = _spins(g), _spins(r)
    nr = r.norm(dim=1)
    return (g - r).norm(dim=1) / torch.maximum(nr, nr.pow(2).mean().sqrt()).clamp_min(1e-300)


def _agree(name, g, r, r32=None, per_spin=True, c=C32):
    """fp64 (r32 None): norm-relative and max_s e_s <= 1e-9.  fp32: norm-relative <= 1e-4 and, per spin,
    e_s <= max(1e-4, c * the reference algorithm's own fp32 e_s).  Every spin the reference moves must move."""
    assert g is not None, name
    assert tuple(g.shape) == tuple(r.shape), (name, tuple(g.shape), tuple(r.shape))
    e = rel(g, r)
    if not per_spin:
        assert e <= (1e-9 if r32 is None else 1e-4), (name, e)
        return
    es = _es(g, r)
    if r32 is None:
        assert e <= 1e-9 and float(es.max()) <= 1e-9, (name, e, float(es.max()), int(es.argmax()))
    else:
        floor = _es(r32, r)
        over = es > 1e-4
        print(f'[fp32 {name}] rel {e:.1e} max e_s {float(es.max()):.1e} (ref fp32 {float(floor.max()):.1e}) '
              f'max e_s/e32_s {float((es / floor.clamp_min(1e-300)).max()):.2f} '
              f'over 1e-4: {float((es[over] / floor[over].clamp_min(1e-300)).max()) if over.any() else 0:.2f}')
        assert e <= 1e-4, (name, e)
        bad = es > torch.clamp(c * floor, min=1e-4)
        assert not bad.any(), (name, 'spins', bad.nonzero().reshape(-1)[:8].tolist(), float(es.max()))
    moved = _spins(r).norm(dim=1) > 0
    still = moved & (_spins(g).norm(dim=1) == 0)
    assert not still.any(), (name, 'spins without a gradient', still.nonzero().reshape(-1)[:8].tolist())


_BWD_LINE = re.compile(r'fused_bwd<(f32|f64),NC=(\d+),PK=(\d+),BLK=(\d+),(precise|fast),ROWS=(\d+),SG=(\d)> '
                       r'grid=\((\d+),(\d+)\) tiles=(\d+) occ=(\d+)')


def _bwd_lines(capfd):
    """The backward launches MRPHY_B200_DEBUG reported since the last read."""
    keys = ('dtype', 'NC', 'PK', 'BLK', 'pol', 'ROWS', 'SG', 'P', 'N', 'tiles', 'occ')
    return [{k: (v if k in ('dtype', 'pol') else int(v)) for k, v in zip(keys, m.groups())}
            for m in _BWD_LINE.finditer(capfd.readouterr().err)]


def _kernel(dtype, nC, wave, policy=None, has_b1=True, pk1=False):
    """The SG instantiation a case must land on: coils rounded up to 1/2/4/8/16 held in registers; fp32 1 and 2 coils pack
    two spins per thread (2 coils: unless MRPHY_B200_NC2_PACK_BWD=1); fp64 ('strict' included) is labelled fast; 'mixed'
    runs a fast backward; ROWS=0 exactly when neither rf nor gr requires grad."""
    is32 = dtype == f32 and policy != 'strict'
    nc = max(nC, 1) if has_b1 else 1
    NC = next(c for c in (1, 2, 4, 8, 16) if nc <= c)
    return dict(dtype='f32' if is32 else 'f64', NC=NC, PK=2 if is32 and (NC == 1 or (NC == 2 and not pk1)) else 1,
                pol='precise' if is32 and (policy or 'precise') == 'precise' else 'fast', ROWS=3 if wave else 0, SG=1)


def _spin_case(dev, capfd, p, dtype, want, K=16, rf=True, gr=None, spin=SPIN, policy=None, sub=None):
    """One SG backward (MRPHY_B200_DEBUG set by the caller) -> its debug line, after checking that it ran `want`; Mo, dL/dM0,
    dL/drf, dL/dgr bitwise as without per-spin gradients; all of them and every per-spin gradient asked for against the
    oracle (dL/drf, dL/dgr only on the whole problem), the others None."""
    gr = rf if gr is None else gr
    capfd.readouterr()
    Mo, g = _fused(p, dev, dtype, K, rf_grad=rf, gr_grad=gr, spin=spin, m0_grad=True, policy=policy, sub=sub)
    lines = [l for l in _bwd_lines(capfd) if l['SG'] == 1]
    assert len(lines) == 1, lines
    assert {k: lines[0][k] for k in want} == want, (lines[0], want)
    with capfd.disabled():
        print('[kernel]', lines[0])
    Mo0, g0 = _fused(p, dev, dtype, K, rf_grad=rf, gr_grad=gr, spin=(), m0_grad=True, policy=policy, sub=sub)
    assert not any(l['SG'] for l in _bwd_lines(capfd))
    assert torch.equal(Mo, Mo0)
    for k, on in (('M0', True), ('rf', rf), ('gr', gr)):
        assert (g[k] is None) == (not on) and (g0[k] is None) == (not on), k
        if on:
            assert torch.equal(g[k], g0[k]), k
    (Mo_r, ref), r32 = _refs(p, dtype, sub)
    c = C32_MUFU if policy in ('fast', 'mixed') else C32
    _agree('Mo', Mo, Mo_r, None if r32 is None else r32[0], c=c)
    for k in ('M0',) + SPIN + ('rf', 'gr'):
        if k in SPIN and (k not in spin or p[k] is None or (k == 'gam' and p['df'] is None)):
            assert g[k] is None, k
        elif k in ('rf', 'gr') and not (rf if k == 'rf' else gr):
            assert g[k] is None, k
        elif k in ('rf', 'gr') and sub is not None:
            continue
        else:
            _agree(k, g[k], ref[k], None if r32 is None else r32[1][k], per_spin=k not in ('rf', 'gr'), c=c)
    return lines[0]


_NC_COILS = {1: 1, 2: 2, 4: 3, 8: 8, 16: 13}   # coils per register class: ragged (3, 13) and full (1, 2, 8)
_KERNELS = [('f32', nc, pk, pol, relax, rows) for nc, pk in ((1, 2), (2, 2), (2, 1), (4, 1), (8, 1), (16, 1))
            for pol in ('precise', 'fast') for relax in (True, False) for rows in (0, 3)] + \
           [('f64', nc, 1, 'fast', relax, rows) for nc in (1, 2, 4, 8, 16) for relax in (True, False) for rows in (0, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize('kern', _KERNELS, ids=[f'{d}-NC{nc}-PK{pk}-{pol}-{"relax" if rl else "norelax"}-rows{r}'
                                                for d, nc, pk, pol, rl, r in _KERNELS])
def test_every_spin_grad_kernel(dev, capfd, monkeypatch, kern):
    """All 68 SG instantiations of fused_bwd_kernel, each asserted from its debug line.  N = 2 with a dt and γ per entry /
    spin; nM = 261, ragged against the 256-spin packed and the 128-spin generic tile; nT = 203 at K = 16: 13 chunks, the
    last partial; 5 spins per entry with b1 = 0 (identity frame), a non-zero b1 phase elsewhere (frame -> lab in sg_fold)."""
    d, NC, PK, pol, relax, rows = kern
    dtype = f32 if d == 'f32' else f64
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    if dtype == f32 and NC == 2 and PK == 1:
        monkeypatch.setenv('MRPHY_B200_NC2_PACK_BWD', '1')
    p = _problem(900 + NC + 50 * relax, 2, 261, 203, _NC_COILS[NC], relax=relax, zero_b1=5)
    _spin_case(dev, capfd, p, dtype, _kernel(dtype, _NC_COILS[NC], rows, pol if dtype == f32 else None, pk1=PK == 1 and NC == 2),
               rf=rows != 0, policy=pol if dtype == f32 else None)


# (id, dtype, nC, problem shape (N, nM, nT), keyword arguments of _spin_case)
_VARIANTS = [(f'{tag}-{w}', dt, nC, (2, 261, 203), dict(rf=w == 'rf', gr=w == 'gr'))
             for tag, dt, nC in (('f32-nC1', f32, 1), ('f32-nC2', f32, 2), ('f32-nC8', f32, 8), ('f64-nC1', f64, 1),
                                 ('f64-nC4', f64, 4)) for w in ('rf', 'gr')] + \
            [(f'{tag}-only-{k}', dt, nC, (2, 261, 203), dict(spin=(k,), rf=False))
             for tag, dt, nC in (('f32-nC1', f32, 1), ('f32-nC8', f32, 8), ('f64-nC4', f64, 4)) for k in SPIN] + \
            [('f32-nC1-default-ckpt', f32, 1, (2, 261, 97), dict(K=None)), ('f64-nC2-default-ckpt', f64, 2, (2, 261, 97), dict(K=None))] + \
            [(f'f32-nC{nC}-{pol}', f32, nC, (2, 261, 203), dict(policy=pol)) for nC in (1, 2, 8) for pol in ('mixed', 'strict')] + \
            [('f32-nC1-nM1', f32, 1, (2, 1, 203), {}), ('f64-nC4-nM1', f64, 4, (2, 1, 203), {}),
             ('f32-nC1-nT1', f32, 1, (2, 261, 1), {}), ('f32-nC8-nT1-fixed', f32, 8, (2, 261, 1), dict(rf=False)),
             ('f32-nC1-N70', f32, 1, (70, 3, 203), {}), ('f64-nC4-N70-fixed', f64, 4, (70, 3, 203), dict(rf=False))]


@pytest.mark.gpu
@pytest.mark.parametrize('case', _VARIANTS, ids=[v[0] for v in _VARIANTS])
def test_spin_grad_kernel_variants(dev, capfd, monkeypatch, case):
    """On a subset of the kernels: one waveform gradient only (ROWS=3, the finalize skips rows; the other is None); each
    spin input on its own (the null outputs of sg_fold); the default checkpoint interval (fp32 single coil: one 128-step
    chunk, first and last at once); 'mixed' and 'strict' per coil family; nM = 1 (a packed pair with a padding spin),
    nT = 1, N = 70 with nM = 3."""
    name, dtype, nC, (N, nM, nT), kw = case
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    p = _problem(500 + len(name), N, nM, nT, nC, zero_b1=1 if nM > 1 else 0)
    kw = dict(kw)
    wave = kw.get('rf', True) or kw.get('gr', False)
    want = _kernel(dtype, nC, wave, kw.get('policy'))
    _spin_case(dev, capfd, p, dtype, want, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize('sched', ['1', '2'])
@pytest.mark.parametrize('rows', [0, 3])
@pytest.mark.parametrize('dtype', [f32, f64])
@pytest.mark.parametrize('nC', [1, 2, 8])
def test_spin_grads_multi_tile(dev, capfd, monkeypatch, nC, dtype, rows, sched):
    """MRPHY_B200_MAX_CTAS=6 on N = 2: 3 CTAs per entry walk 4 to 12 tiles each -- sg_fold's first / last chunk across
    tiles, the per-chunk reset of the sums, the single barrier per chunk of ROWS = 0 at a tile boundary."""
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    monkeypatch.setenv('MRPHY_B200_MAX_CTAS', '6')
    monkeypatch.setenv('MRPHY_B200_SCHED', sched)
    p = _problem(300 + nC, 2, 1500, 97, nC, zero_b1=3)
    line = _spin_case(dev, capfd, p, dtype, _kernel(dtype, nC, rows), rf=rows != 0)
    assert line['tiles'] > line['P'], line


@pytest.mark.gpu
@pytest.mark.parametrize('rows', [0, 3])
def test_spin_grads_sm_aware_grid(dev, capfd, monkeypatch, rows):
    """The default backward grid of one batch entry: c CTAs on every SM with SM-aware tile ownership and its sweep, each
    CTA over many 256-spin tiles (2 x 148 x 8 tiles: more than the resident slots at any occupancy up to 16).  Checked on
    the first tile, the last (partial) tile and 512 seeded spins; dL/drf, dL/dgr bitwise as without per-spin gradients."""
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    tile = 256
    nM = 2 * sms * 8 * tile - 100
    p = _problem(88, 1, nM, 40, 1, zero_b1=3)
    last = (nM - 1) // tile * tile
    gen = torch.Generator().manual_seed(9)
    sub = torch.cat([torch.arange(tile), torch.arange(last, nM), torch.randperm(nM, generator=gen)[:512]]).unique()
    line = _spin_case(dev, capfd, p, f32, _kernel(f32, 1, rows), rf=rows != 0, sub=sub)
    assert line['P'] % sms == 0 and line['P'] > sms and line['tiles'] > line['P'], (line, sms)


_BCAST = {   # name: (input, leaf from the full fp64 value, the leaf expanded to what the oracle sees, nC, state dtype)
    'df_1xM': ('df', lambda x: x[:1], lambda l: l.expand(2, -1), 1, f64),
    'df_transposed': ('df', lambda x: x.t().contiguous().t(), lambda l: l, 1, f64),
    'gam_scalar': ('gam', lambda x: x[0, 0], lambda l: l.expand(2, 150), 1, f64),
    'gam_N': ('gam', lambda x: x[:, 0], lambda l: l[:, None].expand(-1, 150), 1, f64),
    'gam_NxMx1': ('gam', lambda x: x[..., None], lambda l: l[..., 0], 1, f64),
    'gam_f32': ('gam', lambda x: x.float(), lambda l: l.double(), 1, f32),
    'b1_1xM_nC1': ('b1', lambda x: x[:1], lambda l: l.expand(2, -1, -1, -1), 1, f64),
    'b1_1xM_nC4': ('b1', lambda x: x[:1], lambda l: l.expand(2, -1, -1, -1), 4, f64),
    'b1_3d': ('b1', lambda x: x[..., 0], lambda l: l[..., None], 1, f64),
    'loc_expanded': ('loc', lambda x: x[:1], lambda l: l.expand(2, -1, -1), 1, f64),
}


@pytest.mark.gpu
@pytest.mark.parametrize('route', ['op', 'spinarray'])
@pytest.mark.parametrize('case', list(_BCAST))
def test_spin_input_broadcasts(dev, route, case):
    """Spin inputs of a broadcast shape, a non-contiguous Δf and an fp32 γ, through fused_applypulse and SpinArray.applypulse:
    each .grad has its leaf's shape and dtype and equals the oracle's per-spin gradient pushed back through the same
    expansion by autograd."""
    from mrphy import _ops, mobjs
    key, make, grow, nC, dtype = _BCAST[case]
    N, nM, nT = 2, 150, 60
    p = _problem(700 + nC, N, nM, nT, nC, zero_b1=2)
    leaf0 = make(p[key])
    q = dict(p, **{key: grow(leaf0).contiguous()})                     # what the kernels see, in full
    (Mo_r, ref), r32 = _refs(q, dtype)
    lr = leaf0.clone().requires_grad_(True)
    torch.autograd.backward(grow(lr).double(), ref[key])
    want = lr.grad
    kw = {'dtype': dtype, 'device': dev}
    t = {k: (None if v is None else v.to(**kw)) for k, v in p.items()}
    t['gam'], t['dt'] = p['gam'].to(dev), p['dt'].to(dev)
    leaf = make(p[key]).to(dev)
    leaf = (leaf.to(dtype) if key != 'gam' else leaf).detach().requires_grad_(True)
    assert case != 'df_transposed' or not leaf.is_contiguous()
    t[key] = leaf
    loc = t['loc'].expand(N, nM, 3) if key == 'loc' else t['loc']
    if route == 'op':
        Mo = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], loc, Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'], T2_=t['T2'],
                                   γ_=t['gam'], dt=t['dt'])
    else:   # SpinArray keeps γ_ as (N, nM) or broadcastable to it: (N,) and (N, nM, 1) enter as views of the leaf
        gam = t['gam'][:, None] if case == 'gam_N' else t['gam'][..., 0] if case == 'gam_NxMx1' else t['gam']
        sp = mobjs.SpinArray((N, nM), T1_=t['T1'], T2_=t['T2'], γ_=gam, M_=t['M0'], **kw)
        pulse = mobjs.Pulse(rf=t['rf'], gr=t['gr'], dt=t['dt'], **kw)
        Mo = sp.applypulse(pulse, loc_=loc, Δf_=t['df'], b1Map_=t['b1'])
    (Mo * t['w']).sum().backward()
    assert leaf.grad is not None and leaf.grad.shape == leaf.shape and leaf.grad.dtype == leaf.dtype
    w32 = None
    if r32 is not None:
        l32 = leaf0.clone().requires_grad_(True)
        torch.autograd.backward(grow(l32).double(), r32[1][key])
        w32 = l32.grad
    _agree(case, leaf.grad, want, w32)


@pytest.mark.gpu
@pytest.mark.parametrize('route', ['op', 'spinarray'])
def test_gamma_without_df_gets_none(dev, route):
    """γ reaches the loss only through Δf/γ: without Δf its gradient is None, as upstream's autograd leaves it."""
    from mrphy import _ops, mobjs
    p = _problem(31, 1, 40, 30, 1)
    kw = {'dtype': f64, 'device': dev}
    t = {k: (None if v is None else v.to(**kw)) for k, v in p.items()}
    gam, loc = t['gam'].requires_grad_(True), t['loc'].requires_grad_(True)
    if route == 'op':
        Mo = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], loc, b1Map_=t['b1'], T1_=t['T1'], T2_=t['T2'], γ_=gam, dt=t['dt'])
    else:
        sp = mobjs.SpinArray((1, 40), T1_=t['T1'], T2_=t['T2'], γ_=gam, M_=t['M0'], **kw)
        Mo = sp.applypulse(mobjs.Pulse(rf=t['rf'], gr=t['gr'], dt=t['dt'], **kw), loc_=loc, b1Map_=t['b1'])
    (Mo * t['w']).sum().backward()
    assert gam.grad is None and loc.grad is not None


@pytest.mark.gpu
@pytest.mark.parametrize('nC', [1, 4])
@pytest.mark.parametrize('dtype', [f64, f32])
def test_spin_grads_design_route(dev, monkeypatch, dtype, nC):
    """rf = tρθ2rf(ρ, θ, rfmax), gr = s2g(ts2s(ts, smax), dt) with Δf and b1Map requiring grad: the two-stage route (as many
    backward launches as with MRPHY_B200_FUSE_DESIGN=0); dL/dρ, dL/dθ, dL/dts as the fused-design run without per-spin
    gradients (1e-12 / 1e-6 relative, as test_design_adjoint_fused_into_gradient_epilogue); dL/dΔf, dL/db1Map against the
    oracle on the waveforms the kernels were handed."""
    from mrphy import _cabi, _ops, utils
    N, nM, nT = 2, 301, 133
    gen = torch.Generator().manual_seed(41 + nC)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    shp = (N, 1, nT, nC) if nC > 1 else (N, 1, nT)
    d = dict(rho=U(*shp) * 2, theta=U(*shp) * 3, ts=U(N, 3, nT) * 1.5,
             rfmax=(0.15 + 0.05 * U(N, nC).abs()) if nC > 1 else (0.15 + 0.05 * U(N).abs()),
             smax=1.2e4 + 2e3 * U(N, 3).abs(), dt=tensor([4e-6], dtype=f64))
    p = _problem(61 + nC, N, nM, nT, nC)
    kw = {'dtype': dtype, 'device': dev}

    def step(spin, fuse):
        monkeypatch.setenv('MRPHY_B200_FUSE_DESIGN', '1' if fuse else '0')
        v = {k: x.to(**kw) for k, x in d.items()}
        rho, theta, ts = (v[k].requires_grad_(True) for k in ('rho', 'theta', 'ts'))
        rf, gr = utils.tρθ2rf(rho, theta, v['rfmax']), utils.s2g(utils.ts2s(ts, v['smax']), v['dt'])
        t = {k: (None if x is None else x.to(**kw)) for k, x in p.items()}
        df, b1 = t['df'].requires_grad_(spin), t['b1'].requires_grad_(spin)
        Mo = _ops.fused_applypulse(t['M0'], rf, gr, t['loc'], Δf_=df, b1Map_=b1, T1_=t['T1'], T2_=t['T2'],
                                   γ_=p['gam'].to(dev), dt=p['dt'].to(dev))
        n0 = _cabi.launch_counter
        (Mo * t['w']).sum().backward()
        return (rho.grad, theta.grad, ts.grad), (df.grad, b1.grad), _cabi.launch_counter - n0, (rf.detach(), gr.detach())

    g_s, (gdf, gb1), n_s, (rf, gr) = step(True, True)
    g_u, _, n_u, _ = step(True, False)
    g_f, none, _, _ = step(False, True)
    assert none == (None, None)
    assert n_s == n_u, (n_s, n_u)
    for a, b, c in zip(g_s, g_u, g_f):
        assert rel(a, b) < (1e-12 if dtype == f64 else 1e-6)
        assert rel(a, c) < (1e-12 if dtype == f64 else 1e-6)
    q = dict(p, rf=rf.cpu().double(), gr=gr.cpu().double())
    (_, ref), r32 = _refs(q, dtype)
    _agree('df', gdf, ref['df'], None if r32 is None else r32[1]['df'])
    _agree('b1', gb1, ref['b1'], None if r32 is None else r32[1]['b1'])


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [f64, f32])
def test_spin_grads_shard_spins(dev, dtype):
    """parallel.shard_spins with per-spin gradients, both ranks of a world of 2 one after the other on this GPU: the ranks'
    loc_, Δf_, b1Map_, γ_ gradients together are the unsharded ones (not bitwise: the large-angle guard is warp-uniform);
    a Δf_ / γ_ broadcast over spins gets on each rank the sum over that rank's spins, as documented."""
    from mrphy import mobjs, parallel
    N, nM, nT = 2, 1001, 80
    p = _problem(12, N, nM, nT, 1)
    kw = {'dtype': dtype, 'device': dev}
    t = {k: (None if v is None else v.to(**kw)) for k, v in p.items()}
    pulse = mobjs.Pulse(rf=t['rf'], gr=t['gr'], dt=p['dt'].to(dev), **kw)
    tol = 1e-12 if dtype == f64 else 1e-6

    def leaves(bcast):
        x = {k: t[k].clone().requires_grad_(True) for k in ('loc', 'b1')}
        x['df'] = (t['df'][:, :1] if bcast else t['df']).clone().requires_grad_(True)
        x['gam'] = (t['gam'][:, :1] if bcast else t['gam']).to(dtype).clone().requires_grad_(True)
        return x

    def spins(x):
        return mobjs.SpinArray((N, nM), T1_=t['T1'], T2_=t['T2'], γ_=x['gam'], M_=t['M0'], **kw)

    for bcast in (False, True):
        whole = leaves(bcast)
        if bcast:   # the per-spin reference of a broadcast value
            whole = {k: (v.detach().expand(N, nM).clone().requires_grad_(True) if k in ('df', 'gam') else v)
                     for k, v in whole.items()}
        M = spins(whole).applypulse(pulse, loc_=whole['loc'], Δf_=whole['df'], b1Map_=whole['b1'])
        (M * t['w']).sum().backward()
        shard = leaves(False)
        for rank in range(2):
            x = leaves(True) if bcast else shard
            sp, kws = parallel.shard_spins(spins(x), rank, 2, loc_=x['loc'], Δf_=x['df'], b1Map_=x['b1'])
            lo, hi = parallel.shard_range(nM, rank, 2)
            Ml = sp.applypulse(pulse, **kws)
            (Ml * t['w'][:, lo:hi]).sum().backward()
            if bcast:
                for k in ('df', 'gam'):
                    assert x[k].grad.shape == (N, 1)
                    assert rel(x[k].grad, whole[k].grad[:, lo:hi].sum(1, keepdim=True)) < tol, (k, rank)
                for k in ('loc', 'b1'):
                    assert rel(x[k].grad[:, lo:hi], whole[k].grad[:, lo:hi]) < tol, (k, rank)
        if not bcast:
            for k in SPIN:
                assert rel(shard[k].grad, whole[k].grad) < tol, k


# ---- no GPU needed ----------------------------------------------------------------------------------------------------
def test_spin_grad_fields_keep_their_offsets():
    from mrphy import _cabi
    L = _cabi.lib()
    F, P = _cabi.FusedArgs, ctypes.sizeof(ctypes.c_void_p)
    assert L.mrphy_sizeof_args(1) == ctypes.sizeof(F)
    assert (F.gloc.offset, F.gsz.offset, F.gb1.offset) == (F.gMt.offset + P, F.gMt.offset + 2 * P, F.gMt.offset + 3 * P)
    assert L.mrphy_abi_version() == _cabi.ABI_VERSION == 8
    assert 'mrphy_blochsim_fused_bwd' in _cabi.EXPORTS


@pytest.mark.parametrize('nC,want', [(1, (True, True, True)), (8, (False, True, True)), (0, (True, False, False))])
def test_spin_grad_fake_allocates_implementation_shapes(nC, want):
    from mrphy import _cabi, _ops
    N, nM, nT = 2, 37, 50
    e = lambda *s: torch.empty(s, device='meta')
    rf = e(N, 2, nT, nC) if nC else e(N, 2, nT)
    out = _ops._fake_blochsim_fused_bwd(e(N, nM, 3), None, e(N, nM, 3), e(10), e(10), rf, e(N, 3, nT), e(N, nM, 3),
                                        e(N, nM), e(N, nM, 2, max(nC, 1)), None, None, e(1, 1), e(1), 16,
                                        _cabi.FLAG_NEED_GMI, 0, *want, *(None,) * 6, 0, 0)
    gMi, flat, gloc, gsz, gb1 = out[:5]
    assert gMi.shape == (N, nM, 3)
    assert flat.shape == (rf.numel() + N * 3 * nT + _ops.GRAD_TAIL,)
    assert gloc.shape == ((N, nM, 3) if want[0] else (0,))
    assert gsz.shape == ((N, nM) if want[1] else (0,))
    assert gb1.shape == ((N, nM, 2, max(nC, 1)) if want[2] else (0,))


@pytest.mark.parametrize('shape', [(), (1,), (3,), (1, 1), (1, 5), (3, 1), (3, 5), (3, 5, 1), (1, 5, 1), (3, 1, 1), (1, 1, 1),
                                   (3, 5, 1, 1), 'transposed', 'f32'])
def test_param_strides_match_gradient_reduction(shape):
    """Every per-spin constant shape `_param` accepts, at N = 3, nM = 5: the element strides it hands the kernel read the
    broadcast value at every (n, m) and are zero on exactly the axes `_as_param_grad` sums over, and that reduction is
    autograd's of the broadcast (shape and dtype of the input)."""
    from mrphy import _ops
    N, nM = 3, 5
    gen = torch.Generator().manual_seed(1)
    if shape == 'transposed':
        x = torch.rand(nM, N, generator=gen, dtype=f64).t()
    elif shape == 'f32':
        x = torch.rand(N, nM, generator=gen, dtype=f64).float()
    else:
        x = torch.rand(shape, generator=gen, dtype=f64)
    x.requires_grad_(True)
    v = x                                       # the broadcast written out: drop trailing singletons, then (N|1, nM|1)
    while v.ndim > 2:
        v = v[..., 0]
    v = v.reshape(1, 1) if v.ndim == 0 else v[:, None] if v.ndim == 1 else v
    full = v.expand(N, nM)
    p = _ops._param(x, N, nM)
    off = (p.ptr - x.untyped_storage().data_ptr()) // x.element_size()
    read = torch.as_strided(x.detach(), (N, nM), (p.sn, p.sm), off)
    assert torch.equal(read, full.detach())
    assert p.f64 == (x.dtype == f64)
    summed = [v.shape[0] == 1, v.shape[1] == 1]  # the axes _as_param_grad reduces
    assert [p.sn == 0, p.sm == 0] == summed, (p.sn, p.sm, summed)
    g = torch.rand(N, nM, generator=gen, dtype=f64)
    red = _ops._as_param_grad(g, x)
    want, = torch.autograd.grad((full.double() * g).sum(), x)
    assert red.shape == x.shape and red.dtype == x.dtype == want.dtype
    assert torch.allclose(red, want, rtol=1e-6 if x.dtype == f32 else 1e-14, atol=0)
