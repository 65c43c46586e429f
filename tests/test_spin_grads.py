"""Per-spin gradients (loc, Δf, b1Map, γ) from the fused backward, against the fp64 oracle, the explicit-field route and
finite differences; the C-ABI mirror and the fake of the new op need no GPU."""
import ctypes

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


def _oracle(p):
    """dL/d(loc, Δf, b1Map, γ) and Mo of L = sum(w * Mo): dL/dBeff from the oracle's adjoint, then autograd of the field."""
    from oracle import bloch_oracle as orc
    leaves = {k: p[k].clone().requires_grad_(True) for k in ('loc', 'df', 'b1', 'gam') if p[k] is not None}
    q = dict(p, **leaves)
    B = _beff(q['rf'], q['gr'], q['loc'], q['df'], q['b1'], q['gam'])
    assert torch.allclose(B.detach(), orc.rfgr2beff(p['rf'], p['gr'], p['loc'], p['df'], p['b1'], gamma=p['gam']), atol=1e-12)
    Mo, _, gB = orc.blochsim_adj(p['M0'], B.detach(), p['w'], p['T1'], p['T2'], gamma=p['gam'], dt=p['dt'])
    (B * gB).sum().backward()
    return Mo, {k: v.grad for k, v in leaves.items()}


def _fused(p, dev, dtype, K=None, flags=None, rf_grad=True):
    """fused_applypulse with every spin input requiring grad -> (Mo, grads of loc, df, b1, gam, rf, gr)."""
    from mrphy import _ops
    kw = {'dtype': dtype, 'device': dev}
    t = {k: (None if v is None else v.to(**kw)) for k, v in p.items()}
    t['gam'], t['dt'] = p['gam'].to(dev), p['dt'].to(dev)             # fp64 constants next to fp32 state
    leaves = [k for k in ('loc', 'df', 'b1', 'gam') if t[k] is not None] + (['rf', 'gr'] if rf_grad else [])
    for k in leaves:
        t[k].requires_grad_(True)
    Mo = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'],
                               T2_=t['T2'], γ_=t['gam'], dt=t['dt'], ckpt=K, flags=flags)
    (Mo * t['w']).sum().backward()
    return Mo.detach(), {k: t[k].grad for k in leaves}


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
    # a sequence with a gap: the same Δf_ gradient as the explicit route (freeprec adds none, as upstream)
    sp = mobjs.SpinArray((1, 64), **kw)
    loc, dfl = U(1, 64, 3) * 5, U(1, 64) * 100
    gap = tensor(1e-3, dtype=f64)
    grads = []
    for explicit in (False, True):
        d = dfl.clone().requires_grad_(True)
        if explicit:
            M = sp.M_
            for ev in (pulse, gap, pulse):
                M = sims.freeprec(M, gap.to(dev), T1=sp.T1_, T2=sp.T2_, Δf=d) if ev is gap else \
                    sims.blochsim(M, sp.pulse2beff(ev, loc_=loc, Δf_=d), T1=sp.T1_, T2=sp.T2_, γ=sp.γ_, dt=ev.dt)
        else:
            M = sp.applysequence([pulse, gap, pulse], loc_=loc, Δf_=d)
        M.sum().backward()
        grads.append(d.grad)
    assert rel(grads[0], grads[1]) < 1e-9


@pytest.mark.gpu
def test_scale_memory(dev):
    """128³ spins x 2000 steps, fp32: Δf_ and b1Map_ gradients cost at most 1.1x the memory of the rf/gr-only step + 256 MB
    (the dense field and its gradient would need ~100 GB)."""
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
        if spin:
            assert torch.isfinite(df.grad).all() and torch.isfinite(b1.grad).all()
        del Mo
        rf.grad = gr.grad = None
    assert peaks[1] <= 1.1 * peaks[0] + 256 * 2 ** 20, peaks


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


# ---- no GPU needed ----------------------------------------------------------------------------------------------------
def test_spin_grad_args_mirror_matches_library():
    from mrphy import _cabi
    L = _cabi.lib()
    assert L.mrphy_sizeof_args(10) == ctypes.sizeof(_cabi.SpinGradArgs) == 3 * ctypes.sizeof(ctypes.c_void_p)
    assert L.mrphy_abi_version() == _cabi.ABI_VERSION == 6
    assert 'mrphy_blochsim_fused_bwd_spin' in _cabi.EXPORTS


@pytest.mark.parametrize('nC,want', [(1, (True, True, True)), (8, (False, True, True)), (0, (True, False, False))])
def test_fake_allocates_implementation_shapes(nC, want):
    from mrphy import _cabi, _ops
    N, nM, nT = 2, 37, 50
    e = lambda *s: torch.empty(s, device='meta')
    rf = e(N, 2, nT, nC) if nC else e(N, 2, nT)
    out = _ops._fake_blochsim_fused_bwd_spin(e(N, nM, 3), e(N, nM, 3), e(10), e(10), rf, e(N, 3, nT), e(N, nM, 3), e(N, nM),
                                            e(N, nM, 2, max(nC, 1)), None, None, e(1, 1), e(1), 16, _cabi.FLAG_NEED_GMI, *want)
    gMi, flat, gloc, gsz, gb1 = out
    assert gMi.shape == (N, nM, 3)
    assert flat.shape == (rf.numel() + N * 3 * nT + _ops.GRAD_TAIL,)
    assert gloc.shape == ((N, nM, 3) if want[0] else (0,))
    assert gsz.shape == ((N, nM) if want[1] else (0,))
    assert gb1.shape == ((N, nM, 2, max(nC, 1)) if want[2] else (0,))
