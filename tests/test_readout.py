"""The receive signal summed over spins inside the fused kernels (`readout=`): against an einsum over the recorded states of
the same inputs, against the fp64 oracle, gradients against autograd through the record route, bitwise reproducibility,
graph capture and memory at scale; the C-ABI mirror, the refusals, the fakes and the argument checks need no GPU."""
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


def _problem(seed, N, nM, nT, nC, nRx, relax=True, rx_bcast=None):
    """Seeded fp64 inputs; nC = 0: rf without a coil dimension and no b1Map; nRx = 0: no receive map, -1: a map without the
    coil dimension.  rx_bcast 'N' / 'spins': the map is a stride-0 broadcast over that axis."""
    gen = torch.Generator().manual_seed(seed)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    p = dict(rf=U(N, 2, nT, nC) * 0.1 if nC else U(N, 2, nT) * 0.1, gr=U(N, 3, nT) * 2, loc=U(N, nM, 3) * 12,
             df=U(N, nM) * 200, b1=None, M0=torch.nn.functional.normalize(U(N, nM, 3), dim=-1),
             gam=4257.6 * (1 + 0.02 * U(N, nM)), dt=4e-6 * (1 + 0.25 * U(N).abs()),
             T1=(1.0 + 0.5 * U(N, nM)) if relax else None, T2=(0.06 + 0.05 * U(N, nM)) if relax else None, rx=None)
    if nC:
        b1 = U(N, nM, 2, nC) * 0.3
        b1[:, :, 0] += 1
        p['b1'] = b1
    if nRx:
        k = max(nRx, 1)
        shape = (1 if rx_bcast == 'N' else N, 1 if rx_bcast == 'spins' else nM, 2, k)
        rx = U(*shape)
        p['rx'] = rx if nRx > 0 else rx[..., 0]
        p['rx_bcast'] = rx_bcast
    return p


def _leaves(p, dev, dtype, grads):
    kw = {'dtype': dtype, 'device': dev}
    t = {k: (None if (v is None or k == 'rx_bcast') else v.to(**kw)) for k, v in p.items()}
    t['gam'], t['dt'] = p['gam'].to(dev), p['dt'].to(dev)
    for k in grads:
        t[k].requires_grad_(True)
    rx = t['rx']
    if rx is not None and p.get('rx_bcast'):
        N, nM = p['loc'].shape[:2]
        rx = rx.expand((N, nM) + tuple(rx.shape[2:]))          # stride 0: no copy
    return t, rx


def _einsum_signal(Mt, rx):
    """S (N, 2, nR, nRx) from recorded states Mt (N, nM, nR, 3) and a map rx (N, nM, 2, nRx) (None: 1)."""
    mx, my = Mt[..., 0], Mt[..., 1]
    if rx is None:
        return torch.stack([mx.sum(1), my.sum(1)], 1)[..., None]
    rx = rx if rx.ndim == 4 else rx[..., None]
    cx, cy = rx[:, :, 0], rx[:, :, 1]
    Sx = torch.einsum('nik,nir->nrk', cx, mx) - torch.einsum('nik,nir->nrk', cy, my)
    Sy = torch.einsum('nik,nir->nrk', cx, my) + torch.einsum('nik,nir->nrk', cy, mx)
    return torch.stack([Sx, Sy], 1)


def _run(p, dev, dtype, K, s, route, grads=(), wS=None, wM=None, policy=None):
    """route 'readout': fused_applypulse(readout=s); 'record': record=s and an einsum over Mt.  The loss is
    <wS, S> + <wM, M> (either weight may be None) -> (M, S (N,2,nR,nRx), {leaf: grad})."""
    from mrphy import _ops
    t, rx = _leaves(p, dev, dtype, grads)
    _ops.set_trig_policy(policy)
    try:
        kw = dict(Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'], T2_=t['T2'], γ_=t['gam'], dt=t['dt'], ckpt=K)
        if route == 'readout':
            M, S = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], readout=s, rxMap_=rx, **kw)
            S = S if S.ndim == 4 else S[..., None]
        else:
            M, Mt = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], record=s, **kw)
            S = _einsum_signal(Mt, rx)
        if grads:
            loss = 0
            if wS is not None:
                loss = loss + (S * wS.to(S)).sum()
            if wM is not None:
                loss = loss + (M * wM.to(M)).sum()
            loss.backward()
    finally:
        _ops.set_trig_policy(None)
    return M.detach(), S.detach(), {k: t[k].grad for k in grads}


def _abs_c(p):
    rx = p['rx']
    if rx is None:
        return float(p['loc'].shape[1])
    rx = rx if rx.ndim == 4 else rx[..., None]
    N, nM = p['loc'].shape[:2]
    return float(rx.expand(N, nM, 2, rx.shape[3]).norm(dim=2).sum(1).max())


# name: (dtype, nC, nRx, s, N, nM, nT, policy, bcast)
_CASES = {
    'f32-nC1-pk-rx1': (f32, 1, 1, 1, 1, 300, 120, None, None),
    'f32-nC0-nomap': (f32, 0, 0, 3, 2, 5000, 100, None, None),
    'f32-nC2-pk-rx3': (f32, 2, 3, 7, 1, 1000, 100, None, None),
    'f32-nC8-tc-rx16': (f32, 8, 16, 4, 2, 700, 64, None, None),
    'f32-nC1-rx-nodim': (f32, 1, -1, 9, 1, 257, 100, None, None),
    'f32-nC1-bcastN': (f32, 1, 3, 5, 3, 2000, 60, None, 'N'),
    'f32-nC2-bcast-spins': (f32, 2, 2, 2, 1, 777, 50, None, 'spins'),
    'f32-strict-rx3': (f32, 1, 3, 4, 1, 500, 80, 'strict', None),
    'f64-nC4-rx3': (f64, 4, 3, 6, 2, 600, 80, None, None),
    'f64-nC1-rx16': (f64, 1, 16, 1, 1, 300, 40, None, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(_CASES))
def test_signal_matches_einsum_over_recorded_states(dev, case):
    """The same states summed in two orders: within 2e-6·Σ|c| in fp32, 1e-12 relative in fp64 (and 'strict')."""
    dtype, nC, nRx, s, N, nM, nT, policy, bcast = _CASES[case]
    p = _problem(11, N, nM, nT, nC, nRx, rx_bcast=bcast)
    K = 16
    _, S, _ = _run(p, dev, dtype, K, s, 'readout', policy=policy)
    _, ref, _ = _run(p, dev, dtype, K, s, 'record', policy=policy)
    assert S.shape == ref.shape == (N, 2, nT // s, max(nRx, 1)), (S.shape, ref.shape)
    if dtype == f64:
        assert rel(S, ref) <= 1e-12, rel(S, ref)
    else:
        err = float((S - ref).abs().max())
        assert err <= 2e-6 * _abs_c(p), (err, _abs_c(p))


@pytest.mark.gpu
@pytest.mark.parametrize('dtype,nC,nRx', [(f64, 4, 3), (f32, 1, 1), (f32, 8, 2)])
def test_signal_matches_oracle(dev, dtype, nC, nRx):
    """S against the fp64 oracle's states and an einsum: fp64 1e-12 relative; fp32 within max(1e-5, 2 x the reference
    algorithm's own fp32 error) times Σ|c|."""
    from oracle import bloch_oracle as orc
    p = _problem(5, 1, 400, 200, nC, nRx)
    s = 3
    _, S, _ = _run(p, dev, dtype, 16, s, 'readout')
    q = p if dtype == f64 else {k: (v if (v is None or k in ('gam', 'dt', 'rx_bcast')) else v.float().double())
                                for k, v in p.items()}
    B = orc.rfgr2beff(q['rf'], q['gr'], q['loc'], q['df'], q['b1'], gamma=q['gam'])
    Mo, hist = orc.blochsim_fwd(q['M0'], B, q['T1'], q['T2'], gamma=q['gam'], dt=q['dt'], history=True)
    states = torch.cat([hist[1:], Mo[None]]).permute(1, 2, 0, 3)[:, :, s - 1::s]
    ref = _einsum_signal(states, q['rx'])
    if dtype == f64:
        assert rel(S, ref) <= 1e-12
        return
    B32 = orc.rfgr2beff(q['rf'], q['gr'], q['loc'], q['df'], q['b1'], gamma=q['gam'], dtype=f32)
    _, h32 = orc.blochsim_fwd(q['M0'], B32, q['T1'], q['T2'], gamma=q['gam'], dt=q['dt'], dtype=f32, history=True)
    # hist[j] is the state after j steps, states[:, :, r] the one after (r+1)·s
    own32 = h32[s::s].permute(1, 2, 0, 3).double()
    n = min(own32.shape[2], states.shape[2])
    own = float((own32[:, :, :n] - states[:, :, :n]).abs().max())
    err = float((S.cpu().double() - ref).abs().max())
    assert err <= max(1e-5, 2 * own) * _abs_c(p), (err, own)


def _weights(seed, N, nM, nR, nRx):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(N, 2, nR, nRx, generator=g, dtype=f64) - 0.5, torch.rand(N, nM, 3, generator=g, dtype=f64) - 0.5


# name: (dtype, nC, nRx, s, grads, loss on M too)
_GCASES = {
    'f32-nC1-waveform': (f32, 1, 1, 1, ('M0', 'rf', 'gr', 'rx'), False),
    'f32-nC1-S+M': (f32, 1, 3, 4, ('M0', 'rf', 'gr', 'rx'), True),
    'f32-nC1-spin': (f32, 1, 2, 5, ('rf', 'loc', 'df', 'b1', 'gam', 'rx'), True),
    'f32-nC2-spin': (f32, 2, 2, 3, ('rf', 'gr', 'loc', 'df', 'b1', 'rx'), False),
    'f32-nC8': (f32, 8, 4, 6, ('M0', 'rf', 'gr', 'rx'), True),
    'f32-fixed-pulse': (f32, 1, 3, 2, ('rx',), False),
    'f32-rf-only': (f32, 1, 0, 2, ('rf',), False),
    'f64-nC4-spin': (f64, 4, 3, 5, ('M0', 'rf', 'gr', 'loc', 'df', 'b1', 'gam', 'rx'), True),
    'f64-nC1': (f64, 1, 16, 1, ('M0', 'rf', 'gr', 'rx'), False),
}


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(_GCASES))
def test_gradients_match_record_route(dev, case):
    """Gradients of <wS, S> (+ <wM, M>) against autograd through record + einsum: 1e-4 relative in fp32, 1e-10 in fp64."""
    dtype, nC, nRx, s, grads, on_M = _GCASES[case]
    N, nM, nT = 2, 600, 90
    p = _problem(21, N, nM, nT, nC, nRx)
    grads = tuple(g for g in grads if not (g == 'rx' and p['rx'] is None))
    wS, wM = _weights(3, N, nM, nT // s, max(nRx, 1))
    _, S, g = _run(p, dev, dtype, 16, s, 'readout', grads, wS, wM if on_M else None)
    _, ref, gr_ = _run(p, dev, dtype, 16, s, 'record', grads, wS, wM if on_M else None)
    tol = 1e-4 if dtype == f32 else 1e-10
    for k in grads:
        assert g[k] is not None and g[k].shape == gr_[k].shape, k
        assert rel(g[k], gr_[k]) <= tol, (k, rel(g[k], gr_[k]))


# name: (dtype, nC, nRx, nM, nT, s, MRPHY_B200_MAX_CTAS or None)
_MCASES = {
    'f32-nC1-pk': (f32, 1, 2, 2000, 40, 3, '3'),
    'f32-nC2-pk': (f32, 2, 3, 2000, 40, 2, '3'),
    'f32-nC8-tc': (f32, 8, 3, 2000, 32, 4, '3'),
    'f64-nC4': (f64, 4, 2, 1500, 40, 5, '2'),
    'f32-nC1-300k': (f32, 1, 1, 300000, 20, 1, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(_MCASES))
def test_multi_tile_ctas_match_record_route(dev, capfd, monkeypatch, case):
    """CTAs that own several spin tiles -- the forward's store-then-add into its slot, the backward's per-tile weights, dL/drx
    sums and re-staged dL/dS: S and the gradients of M_, rf, gr, loc and rxMap against record + einsum.  The launch lines
    confirm that every readout kernel ran with more tiles than CTAs (a CTA cap, or 3e5 spins at the default grid)."""
    dtype, nC, nRx, nM, nT, s, cap = _MCASES[case]
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    if cap:
        monkeypatch.setenv('MRPHY_B200_MAX_CTAS', cap)
    p = _problem(31, 1, nM, nT, nC, nRx)
    grads = ('M0', 'rf', 'gr', 'loc', 'rx')
    wS, wM = _weights(6, 1, nM, nT // s, nRx)
    K = 16
    capfd.readouterr()
    _, S, g = _run(p, dev, dtype, K, s, 'readout', grads, wS, wM)
    lines = re.findall(r'(fused_\w+)<[^>]*RD=1> grid=\((\d+),(\d+)\) tiles=(\d+)', capfd.readouterr().err)
    assert {name for name, *_ in lines} >= {'fused_bwd', 'fused_fwd_tc' if nC >= 4 and dtype == f32 else 'fused_fwd'}, lines
    for name, P, N, tiles in lines:
        assert int(tiles) > int(P), (name, P, tiles)          # some CTA owns two tiles or more
    _, ref, gr_ = _run(p, dev, dtype, K, s, 'record', grads, wS, wM)
    if dtype == f64:
        assert rel(S, ref) <= 1e-12, rel(S, ref)
    else:
        err = float((S - ref).abs().max())
        assert err <= 2e-6 * _abs_c(p), (err, _abs_c(p))
    tol = 1e-4 if dtype == f32 else 1e-10
    for k in grads:
        assert rel(g[k], gr_[k]) <= tol, (k, rel(g[k], gr_[k]))


@pytest.mark.gpu
@pytest.mark.parametrize('dtype,nC,nRx', [(f32, 1, 1), (f32, 2, 3), (f32, 8, 16), (f64, 4, 2)])
def test_bitwise_reproducible(dev, dtype, nC, nRx):
    """Two identical calls: S and every gradient are equal bit for bit (multi-tile grid, ragged last tile)."""
    p = _problem(8, 1, 70001, 64, nC, nRx)
    wS, wM = _weights(4, 1, 70001, 64, nRx)
    grads = ('M0', 'rf', 'gr', 'loc', 'rx')
    a = _run(p, dev, dtype, 16, 1, 'readout', grads, wS, wM)
    b = _run(p, dev, dtype, 16, 1, 'readout', grads, wS, wM)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for k in grads:
        assert torch.equal(a[2][k], b[2][k]), k


@pytest.mark.gpu
def test_loss_ignoring_S_is_bitwise_unchanged(dev):
    """A loss on M alone runs the backward without the readout: M and the gradients equal a call without readout."""
    from mrphy import _ops
    p = _problem(9, 1, 3000, 100, 1, 2)
    outs = []
    for readout in (None, 4):
        t, rx = _leaves(p, dev, f32, ('rf', 'gr', 'M0'))
        out = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'],
                                    T2_=t['T2'], γ_=t['gam'], dt=t['dt'], readout=readout, rxMap_=rx if readout else None)
        M = out if readout is None else out[0]
        (M * M).sum().backward()
        outs.append((M.detach(), t['rf'].grad, t['gr'].grad, t['M0'].grad))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_finite_differences_fp64(dev):
    """dL/drxMap and dL/drf against central differences of the fp64 readout."""
    from mrphy import _ops
    p = _problem(13, 1, 50, 30, 1, 2)
    wS, _ = _weights(5, 1, 50, 10, 2)
    wS = wS.to(dev)
    _, _, g = _run(p, dev, f64, 8, 3, 'readout', ('rf', 'rx'), wS, None)

    def loss(q):
        t, rx = _leaves(q, dev, f64, ())
        _, S = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'],
                                     T2_=t['T2'], γ_=t['gam'], dt=t['dt'], ckpt=8, readout=3, rxMap_=rx)
        return float((S * wS).sum())
    h = 1e-6
    for key, idx in (('rx', (0, 7, 1, 1)), ('rx', (0, 31, 0, 0)), ('rf', (0, 0, 4)), ('rf', (0, 1, 20))):
        qp, qm = dict(p), dict(p)
        qp[key], qm[key] = p[key].clone(), p[key].clone()
        qp[key][idx] += h
        qm[key][idx] -= h
        fd = (loss(qp) - loss(qm)) / (2 * h)
        an = float(g[key][idx])
        assert abs(fd - an) <= 1e-6 * max(1.0, abs(fd)), (key, idx, fd, an)


@pytest.mark.gpu
def test_spincube_readout(dev):
    """SpinCube.applypulse(readout=, rxMap=) on a masked cube: S matches the compact call; doEmbed applies to M."""
    from mrphy import mobjs
    kw = {'dtype': f32, 'device': dev}
    mask = torch.zeros(1, 6, 5, 4, dtype=torch.bool)
    mask[:, 1:5, :, 1:] = True
    cube = mobjs.SpinCube((1, 6, 5, 4), tensor([[12., 10., 8.]]), mask=mask, **kw)
    gen = torch.Generator().manual_seed(2)
    rxMap = (torch.rand(1, 6, 5, 4, 2, 3, generator=gen) - 0.5).to(dev)
    pulse = mobjs.Pulse(rf=(torch.rand(1, 2, 40, generator=gen) * 0.1).to(dev), gr=torch.rand(1, 3, 40, generator=gen).to(dev),
                        **kw)
    M, S = cube.applypulse(pulse, readout=5, rxMap=rxMap, doEmbed=True)
    M_, S_ = cube.applypulse(pulse, readout=5, rxMap_=cube.extract(rxMap))
    assert M.shape == (1, 6, 5, 4, 3) and S.shape == (1, 2, 8, 3)
    assert torch.equal(S, S_) and torch.equal(cube.extract(M), M_)


@pytest.mark.gpu
def test_graph_capture_readout(dev):
    from mrphy import graphs, mobjs
    kw = {'dtype': f32, 'device': dev}
    gen = torch.Generator().manual_seed(4)
    U = lambda *s: (torch.rand(s, generator=gen) * 2 - 1).to(dev)
    sp = mobjs.SpinArray((1, 2000), **kw)
    loc = U(1, 2000, 3) * 5
    rx = U(1, 2000, 2, 2).requires_grad_(True)
    pulse = mobjs.Pulse(rf=(U(1, 2, 100) * 0.1).requires_grad_(True), gr=(U(1, 3, 100) * 2).requires_grad_(True), **kw)
    step = graphs.capture(lambda: sp.applypulse(pulse, loc_=loc, readout=2, rxMap_=rx)[1].pow(2).sum().backward(),
                          params=[rx, pulse.rf, pulse.gr])
    step.replay()
    torch.cuda.synchronize()
    first = [rx.grad.clone(), pulse.rf.grad.clone(), pulse.gr.grad.clone()]
    step.replay()
    torch.cuda.synchronize()
    for a, b in zip(first, (rx.grad, pulse.rf.grad, pulse.gr.grad)):
        assert torch.equal(a, b)
    rx2 = rx.detach().clone().requires_grad_(True)
    rf2, gr2 = pulse.rf.detach().clone().requires_grad_(True), pulse.gr.detach().clone().requires_grad_(True)
    sp.applypulse(mobjs.Pulse(rf=rf2, gr=gr2, **kw), loc_=loc, readout=2, rxMap_=rx2)[1].pow(2).sum().backward()
    for a, b in zip(first, (rx2.grad, rf2.grad, gr2.grad)):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_readout_scale_memory(dev):
    """128³ spins x 2000 steps, fp32, s = 1: peak memory at most the step without readout + S + the readout workspace +
    256 MB (the record route would need 2 x 50 GB).  The receive map is zero except on 256 seeded spins, so the full-size
    run's S -- every CTA summing many tiles into its slot -- is those spins' signal, checked against the oracle."""
    from mrphy import _cabi, _ops
    nM, nT, s = 128 ** 3, 2000, 1
    gen = torch.Generator(device=dev).manual_seed(0)
    U = lambda *sh: torch.rand(sh, generator=gen, device=dev) * 2 - 1
    M0 = torch.nn.functional.normalize(U(1, nM, 3), dim=-1)
    loc, df = U(1, nM, 3) * 12, U(1, nM) * 100
    rf, gr = (U(1, 2, nT) * 0.1).requires_grad_(True), (U(1, 3, nT) * 2).requires_grad_(True)
    kw = dict(Δf_=df, γ_=tensor(4257.6, dtype=f64), dt=tensor(4e-6, dtype=f64))
    wS = torch.rand(1, 2, nT, generator=gen, device=dev) - 0.5
    sub = torch.randperm(nM, generator=torch.Generator().manual_seed(3))[:256].to(dev)
    rx = torch.zeros(1, nM, 2, device=dev)
    rx[:, sub] = U(1, 256, 2)
    peaks = []
    for readout in (None, s):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = _ops.fused_applypulse(M0, rf, gr, loc, readout=readout, rxMap_=rx if readout else None, **kw)
        if readout is None:
            out.sum().backward()
        else:
            (out[0].sum() + (out[1] * wS).sum()).backward()
            S = out[1].detach()
        torch.cuda.synchronize()
        peaks.append(torch.cuda.max_memory_allocated() - base)
        del out
        rf.grad = gr.grad = None
    a = _cabi.FusedArgs()
    a.dtype, a.N, a.nM, a.nT, a.nC, a.K, a.every, a.nR, a.nRx = _cabi.MRPHY_F32, 1, nM, nT, 1, 128, s, nT // s, 1
    work = _cabi.lib().mrphy_fused_readout_elems(a) * 4
    assert peaks[1] <= peaks[0] + 2 * nT * 4 + work + 256 * 2 ** 20, (peaks, work)
    c = lambda x: x.detach()[:, sub].cpu().double()
    from oracle import bloch_oracle as orc
    q = dict(rf=rf.detach().cpu().double(), gr=gr.detach().cpu().double(), loc=c(loc), df=c(df), M0=c(M0),
             gam=torch.full((1, 256), 4257.6, dtype=f64), dt=tensor(4e-6, dtype=f64), rx=c(rx))
    B = orc.rfgr2beff(q['rf'], q['gr'], q['loc'], q['df'], None, gamma=q['gam'])
    Mo, hist = orc.blochsim_fwd(q['M0'], B, None, None, gamma=q['gam'], dt=q['dt'], history=True)
    states = torch.cat([hist[1:], Mo[None]]).permute(1, 2, 0, 3)
    ref = _einsum_signal(states, q['rx'])[..., 0]
    B32 = orc.rfgr2beff(q['rf'], q['gr'], q['loc'], q['df'], None, gamma=q['gam'], dtype=f32)
    _, h32 = orc.blochsim_fwd(q['M0'], B32, None, None, gamma=q['gam'], dt=q['dt'], dtype=f32, history=True)
    own = float((h32[1:].permute(1, 2, 0, 3).double() - states[:, :, :-1]).abs().max())
    err = float((S.cpu().double() - ref).abs().max())
    sum_c = float(q['rx'].norm(dim=2).sum())
    assert err <= max(1e-5, 2 * own) * sum_c, (err, own, sum_c)


# ---------------------------------------------------------------------------------------------------------- host only
def test_readout_fields_mirror_matches_library():
    """The readout fields close mrphy_fused_args, behind the design tail; no struct or entry point of their own."""
    from mrphy import _cabi
    L = _cabi.lib()
    F, P = _cabi.FusedArgs, ctypes.sizeof(ctypes.c_void_p)
    assert L.mrphy_sizeof_args(1) == ctypes.sizeof(F) == F.S_work.offset + P
    assert (F.nRx.offset, F.rx.offset) == (F.design.offset + P, F.design.offset + P + 8)
    assert (F.rx_sn.offset, F.rx_sm.offset) == (F.rx.offset + P, F.rx.offset + P + 8)
    assert (F.S.offset, F.gS.offset, F.grx.offset, F.S_work.offset) == tuple(F.rx_sm.offset + 8 + k * P for k in range(4))
    assert L.mrphy_sizeof_args(10) == 0
    assert L.mrphy_abi_version() == _cabi.ABI_VERSION == 8
    assert {'mrphy_blochsim_fused_fwd', 'mrphy_blochsim_fused_bwd', 'mrphy_fused_readout_elems'} <= set(_cabi.EXPORTS)
    assert not {f'mrphy_blochsim_fused_readout_{d}' for d in ('fwd', 'bwd')} & set(_cabi.EXPORTS)   # the former pair


def _refusable_args():
    """FusedArgs whose checks all pass up to the readout's; the pointers are never dereferenced."""
    from mrphy import _cabi
    a = _cabi.FusedArgs()
    a.dtype, a.N, a.nM, a.nT, a.nC, a.K = _cabi.MRPHY_F32, 1, 4, 10, 1, 8
    for p in ('Mi', 'rf', 'gr', 'loc', 'Mo', 'ckpt', 'wave', 'gMo', 'partials', 'grf', 'ggr'):
        setattr(a, p, 256)
    a.gamma.ptr = a.dt.ptr = 256
    a.every, a.nR = 3, 3
    a.nRx, a.S, a.gS, a.S_work = 2, 256, 256, 256
    return a


@pytest.mark.parametrize('bad', ['Mt', 'gMt', 'design', 'nRx0', 'nRx17', 'S', 'work', 'gS', 'every0', 'every11', 'nR'])
def test_fused_entry_points_refuse_bad_readout(bad):
    """Every refusal is MRPHY_ERR_ARG with nothing launched."""
    from mrphy import _cabi
    L = _cabi.lib()
    a = _refusable_args()
    bwd = bad in ('gMt', 'design', 'gS')
    d = _cabi.ReparamArgs()
    if bad in ('Mt', 'gMt'):
        setattr(a, bad, 256)
    elif bad == 'design':
        d.dtype, d.adjoint, d.N, d.nT, d.nC, d.rf_kind = a.dtype, 1, a.N, a.nT, 1, 1
        d.rho = d.theta = d.rfmax = d.grho = d.gtheta = 256
        a.design = ctypes.addressof(d)
    elif bad.startswith('nRx'):
        a.nRx = int(bad[3:])                 # nRx0: S, gS, S_work stay set, so the readout is on and refused
    elif bad in ('S', 'work', 'gS'):
        setattr(a, 'S_work' if bad == 'work' else bad, None)
    elif bad.startswith('every'):
        a.every = int(bad[5:])
    else:
        a.nR = 2
    for b in ((False, True) if bad.startswith(('nRx', 'every', 'nR', 'Mt')) else (bwd,)):
        rc = L.mrphy_blochsim_fused_bwd(a, 1, None) if b else L.mrphy_blochsim_fused_fwd(a, None)
        assert rc == -1, (bad, b, rc)
        assert L.mrphy_last_launch_count() == 0
        assert 'readout' in L.mrphy_last_error().decode()


def test_readout_elems_sizing_from_fused_args():
    from mrphy import _cabi
    L = _cabi.lib()
    a = _refusable_args()
    a.nM, a.nT, a.every, a.nR, a.nRx = 1000, 100, 7, 14, 3
    # ceil(1000 / 128) = 8 CTAs per batch entry at most, one slot [nR][2 nRx] each
    assert L.mrphy_fused_readout_elems(a) == 8 * 14 * 6
    a.nRx = 17
    assert L.mrphy_fused_readout_elems(a) == 0


@pytest.mark.parametrize('nRx', [0, 1, 8])
def test_fused_fakes_allocate_readout_shapes(nRx):
    from mrphy import _cabi, _ops
    N, nM, nT, every, nC = 2, 37, 50, 7, 2
    e = lambda *s: torch.empty(s, device='meta')
    rf, b1 = e(N, 2, nT, nC), e(N, nM, 2, nC)
    rx = e(N, nM, 2, nRx) if nRx else None
    args = (e(N, nM, 3), rf, e(N, 3, nT), e(N, nM, 3), e(N, nM), b1, None, None, e(1, 1), e(1), 16, 0)
    Mo, S, ckpt, wave = _ops._fake_blochsim_fused_fwd(*args, every, max(nRx, 1), rx)
    ref = _ops._fake_blochsim_fused_fwd(*args, 0)
    assert Mo.shape == (N, nM, 3) and S.shape == (N, 2, nT // every, max(nRx, 1))
    assert ckpt.shape == ref[2].shape and wave.shape == ref[3].shape
    for want_rx in (False, True):
        out = _ops._fake_blochsim_fused_bwd(Mo, S, Mo, ckpt, wave, rf, e(N, 3, nT), e(N, nM, 3), e(N, nM), b1, None, None,
                                            e(1, 1), e(1), 16, _cabi.FLAG_NEED_GMI, every, True, True, True, *(None,) * 6, 0,
                                            0, max(nRx, 1), rx, want_rx)
        gMi, flat, gloc, gsz, gb1, *_, grx = out
        assert gMi.shape == (N, nM, 3) and flat.shape == (rf.numel() + N * 3 * nT + _ops.GRAD_TAIL,)
        assert gloc.shape == (N, nM, 3) and gsz.shape == (N, nM) and gb1.shape == (N, nM, 2, nC)
        assert grx.shape == ((N, nM, 2, max(nRx, 1)) if want_rx else (0,))


@pytest.mark.parametrize('kw,match', [(dict(readout=0), 'outside'), (dict(readout=31), 'outside'),
                                      (dict(readout=2.5), 'integer'), (dict(readout=True), 'integer'),
                                      (dict(readout='4'), 'integer'), (dict(readout=3, record=3), 'record'),
                                      (dict(readout=3, nRx=17), '16 receive coils'),
                                      (dict(readout=3, nC=17), '16 transmit coils')])
def test_bad_readout_raises_before_anything_runs(kw, match):
    """ValueError before the device is looked at (CPU tensors here), through fused_applypulse and SpinArray.applypulse."""
    from mrphy import _ops, mobjs
    kw = dict(kw)
    nRx, nC = kw.pop('nRx', 2), kw.pop('nC', 1)
    p = _problem(1, 1, 5, 30, nC, nRx)
    with pytest.raises(ValueError, match=match):
        _ops.fused_applypulse(p['M0'], p['rf'], p['gr'], p['loc'], b1Map_=p['b1'], γ_=p['gam'], dt=p['dt'], rxMap_=p['rx'],
                              **kw)
    sp = mobjs.SpinArray((1, 5), dtype=f64)
    pulse = mobjs.Pulse(rf=p['rf'], gr=p['gr'], dtype=f64)
    with pytest.raises(ValueError, match=match):
        sp.applypulse(pulse, loc_=p['loc'], b1Map_=p['b1'], rxMap_=p['rx'], **kw)
