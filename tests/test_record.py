"""Recording the magnetisation every s steps in the fused kernels (`record=`): prefix identity against truncated pulses,
gradients by linearity, the fp64 oracle, the layers above the op; the C-ABI mirror, the fakes and the refusals need no GPU."""
import ctypes
import os
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


def _problem(seed, N, nM, nT, nC, relax=True):
    """Seeded fp64 inputs with a dt per batch entry and a γ per spin; nC = 0: rf without a coil dimension, no b1Map."""
    gen = torch.Generator().manual_seed(seed)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    p = dict(rf=U(N, 2, nT, nC) * 0.1 if nC else U(N, 2, nT) * 0.1, gr=U(N, 3, nT) * 2, loc=U(N, nM, 3) * 12,
             df=U(N, nM) * 200, b1=None, M0=torch.nn.functional.normalize(U(N, nM, 3), dim=-1),
             gam=4257.6 * (1 + 0.02 * U(N, nM)), dt=4e-6 * (1 + 0.25 * U(N).abs()),
             T1=(1.0 + 0.5 * U(N, nM)) if relax else None, T2=(0.06 + 0.05 * U(N, nM)) if relax else None)
    if nC:
        b1 = U(N, nM, 2, nC) * 0.3
        b1[:, :, 0] += 1
        p['b1'] = b1
    return p


LEAVES = ('M0', 'rf', 'gr', 'loc', 'df', 'b1', 'gam')


def _run(p, dev, dtype, K, nT=None, record=None, grads=(), w=None, wt=None, policy=None):
    """fused_applypulse on the first `nT` samples of the pulse; with `grads` the leaves that require grad and the loss
    <w, M> + sum_r <wt[..., r, :], Mt[..., r, :]> (either weight may be None) -> (M, Mt, {leaf: grad})."""
    from mrphy import _ops
    kw = {'dtype': dtype, 'device': dev}
    nT = p['rf'].shape[2] if nT is None else nT
    t = {k: (None if v is None else v.to(**kw)) for k, v in p.items()}
    t['gam'], t['dt'] = p['gam'].to(dev), p['dt'].to(dev)
    t['rf'], t['gr'] = t['rf'][:, :, :nT].contiguous(), t['gr'][:, :, :nT].contiguous()
    for k in grads:
        t[k].requires_grad_(True)
    _ops.set_trig_policy(policy)
    try:
        out = _ops.fused_applypulse(t['M0'], t['rf'], t['gr'], t['loc'], Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'],
                                    T2_=t['T2'], γ_=t['gam'], dt=t['dt'], ckpt=K, record=record)
        M, Mt = out if record is not None else (out, None)
        if grads:
            loss = 0
            if w is not None:
                loss = loss + (M * w.to(M)).sum()
            if wt is not None:
                loss = loss + (Mt * wt.to(Mt)).sum()
            loss.backward()
    finally:
        _ops.set_trig_policy(None)
    return M.detach(), (None if Mt is None else Mt.detach()), {k: t[k].grad for k in grads}


_FWD_LINE = re.compile(r'fused_fwd(_tc)?<([^>]*)> ')
_BWD_LINE = re.compile(r'fused_bwd<([^>]*)> ')


def _lines(capfd, pat):
    return [m.group(0) for m in pat.finditer(capfd.readouterr().err)]


# kernel families of the forward: (id, dtype, coils (0: no b1Map), env, policy, expected debug-line fragment)
_FAMILIES = [
    ('f32-nC1-packed', f32, 1, {}, 'precise', 'fused_fwd<f32,NC=1,PK=2,BLK=64,precise,REC=1>'),
    ('f32-nC1-fast', f32, 1, {}, 'fast', 'fused_fwd<f32,NC=1,PK=2,BLK=64,fast,REC=1>'),
    ('f32-nC1-mixed', f32, 1, {}, 'mixed', 'fused_fwd<f32,NC=1,PK=2,BLK=64,precise,REC=1>'),
    ('f32-nob1', f32, 0, {}, 'precise', 'fused_fwd<f32,NC=1,PK=2,BLK=64,precise,REC=1>'),
    ('f32-nC2-packed', f32, 2, {}, 'precise', 'fused_fwd<f32,NC=2,PK=2,BLK=64,precise,REC=1>'),
    ('f32-nC3-tc4', f32, 3, {}, 'precise', 'fused_fwd_tc<NC=4,PK=2,REC=1>'),
    ('f32-nC8-tc8', f32, 8, {}, 'fast', 'fused_fwd_tc<NC=8,PK=2,REC=1>'),
    ('f32-nC13-tc16', f32, 13, {}, 'precise', 'fused_fwd_tc<NC=16,PK=2,REC=1>'),
    ('f32-nC4-fma', f32, 4, {'MRPHY_B200_TC': '0'}, 'precise', 'fused_fwd<f32,NC=4,PK=1,BLK=128,precise,REC=1>'),
    ('f64-nC1', f64, 1, {}, None, 'fused_fwd<f64,NC=1,PK=1,BLK=128,fast,REC=1>'),
    ('f64-nC4', f64, 4, {}, None, 'fused_fwd<f64,NC=4,PK=1,BLK=128,fast,REC=1>'),
]
_FAM_IDS = [f[0] for f in _FAMILIES]


@pytest.mark.gpu
@pytest.mark.parametrize('relax', [True, False], ids=['relax', 'norelax'])
@pytest.mark.parametrize('fam', _FAMILIES, ids=_FAM_IDS)
def test_prefix_identity(dev, capfd, monkeypatch, fam, relax):
    """Mt[..., r, :] is bitwise M of the pulse cut to its first (r+1)·s samples, at K = 16 and nT = 45 (chunks 16, 16, 13):
    s = 1, s = 7 (records inside 4-step groups and across chunk boundaries, 45 % 7 != 0), s = 9 (divides nT), s = nT; and
    nT = 1.  nM = 257: one spin past a 256-spin tile."""
    _, dtype, nC, env, pol, frag = fam
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    p = _problem(11 + nC + 100 * relax, 2, 257, 45, nC, relax=relax)
    for nT, s in ((45, 1), (45, 7), (45, 9), (45, 45), (1, 1)):
        capfd.readouterr()
        M, Mt, _ = _run(p, dev, dtype, 16, nT=nT, record=s, policy=pol)
        lines = _lines(capfd, _FWD_LINE)
        assert len(lines) == 1 and frag in lines[0], (lines, frag)
        nR = nT // s
        assert Mt.shape == (2, 257, nR, 3) and Mt.dtype == dtype
        assert not Mt.is_contiguous()
        M0, _, _ = _run(p, dev, dtype, 16, nT=nT, policy=pol)
        assert torch.equal(M, M0)
        assert not any('REC' in l for l in _lines(capfd, _FWD_LINE))
        for r in range(nR):
            Mr, _, _ = _run(p, dev, dtype, 16, nT=(r + 1) * s, policy=pol)
            assert torch.equal(Mt[:, :, r], Mr), (nT, s, r, float((Mt[:, :, r] - Mr).abs().max()))
        if nT % s == 0:
            assert torch.equal(Mt[:, :, -1], M)


def _oracle_states(p, sub=None):
    """fp64 oracle: the state after every step, (N, nM, nT, 3)."""
    from oracle import bloch_oracle as orc
    q = {k: (v if v is None or sub is None or k in ('rf', 'gr', 'dt') else v[:, sub]) for k, v in p.items()}
    B = orc.rfgr2beff(q['rf'], q['gr'], q['loc'], q['df'], q['b1'], gamma=q['gam'])
    Mo, hist = orc.blochsim_fwd(q['M0'], B, q['T1'], q['T2'], gamma=q['gam'], dt=q['dt'], history=True)
    return torch.cat([hist[1:], Mo[None]]).permute(1, 2, 0, 3)


def _as32(p):
    return {k: (None if v is None else (v if k in ('gam', 'dt') else v.float().double())) for k, v in p.items()}


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['f64-nC1', 'f64-nC4', 'f32-nC1', 'f32-nC8', 'f32-strict'])
def test_states_match_oracle(dev, case):
    """Mt against the fp64 oracle's states: 1e-12 in fp64; fp32 within max(1e-5, the reference algorithm's own fp32
    error on the same inputs); 'strict' (fp32 in and out, fp64 inside) within 1e-5."""
    from oracle import bloch_oracle as orc
    dtype = f64 if case.startswith('f64') else f32
    nC = 4 if case == 'f64-nC4' else (8 if case == 'f32-nC8' else 1)
    p = _problem(5, 2, 200, 300, nC)
    M, Mt, _ = _run(p, dev, dtype, 16, record=3, policy='strict' if case == 'f32-strict' else None)
    assert Mt.dtype == dtype
    q = p if dtype == f64 else _as32(p)
    ref = _oracle_states(q)[:, :, 2::3]
    err = float((Mt.cpu().double() - ref).abs().max())
    if dtype == f64:
        assert err <= 1e-12, err
    elif case == 'f32-strict':
        assert err <= 1e-5, err
    else:
        B = orc.rfgr2beff(q['rf'], q['gr'], q['loc'], q['df'], q['b1'], gamma=q['gam'], dtype=f32)
        _, h32 = orc.blochsim_fwd(q['M0'], B, q['T1'], q['T2'], gamma=q['gam'], dt=q['dt'], dtype=f32, history=True)
        own = float((h32[3::3].permute(1, 2, 0, 3).double() - ref[:, :, :-1]).abs().max())
        assert err <= max(1e-5, own), (err, own)


def _linear_reference(p, dev, dtype, K, s, grads, w, wt, policy=None):
    """Gradients of sum_r <wt_r, M(first (r+1)s samples)> + <w, M>, one truncated run per r, rf/gr zero-padded to nT."""
    nT = p['rf'].shape[2]
    tot = {}
    terms = [(nT, w)] + [((r + 1) * s, wt[:, :, r]) for r in range(nT // s)]
    for n, wr in terms:
        if wr is None:
            continue
        _, _, g = _run(p, dev, dtype, K, nT=n, grads=grads, w=wr, policy=policy)
        for k, v in g.items():
            if v is None:
                continue
            if k in ('rf', 'gr'):
                v = torch.nn.functional.pad(v, (0, 0, 0, nT - n) if (k == 'rf' and v.ndim == 4) else (0, nT - n))
            tot[k] = tot[k] + v if k in tot else v.clone()
    return tot


def _weights(seed, N, nM, nT, s, on_M=True, on_Mt=True):
    gen = torch.Generator().manual_seed(seed)
    U = lambda *sh: torch.rand(sh, generator=gen, dtype=f64) * 2 - 1
    return (U(N, nM, 3) if on_M else None), (U(N, nM, nT // s, 3) if on_Mt else None)


def _check_linearity(p, dev, dtype, s, grads, K=16, on_M=True, on_Mt=True, policy=None, capfd=None, frag='REC=1'):
    N, nM, nT = p['M0'].shape[0], p['M0'].shape[1], p['rf'].shape[2]
    w, wt = _weights(7, N, nM, nT, s, on_M, on_Mt)
    if capfd is not None:
        capfd.readouterr()
    _, _, g = _run(p, dev, dtype, K, record=s, grads=grads, w=w, wt=wt, policy=policy)
    if capfd is not None:
        lines = _lines(capfd, _BWD_LINE)
        assert len(lines) == 1 and frag in lines[0], (lines, frag)
    ref = _linear_reference(p, dev, dtype, K, s, grads, w, wt, policy)
    tol = 1e-10 if dtype == f64 and policy != 'strict' else 1e-4
    for k in grads:
        if k == 'gam' and p['df'] is None:
            continue
        assert g[k] is not None and torch.isfinite(g[k]).all(), k
        assert rel(g[k], ref[k]) <= tol, (k, rel(g[k], ref[k]))
    return g


@pytest.mark.gpu
@pytest.mark.parametrize('fam', _FAMILIES, ids=_FAM_IDS)
def test_gradients_by_linearity(dev, capfd, monkeypatch, fam):
    """Gradients of sum_r <w_r, Mt_r> + <w, M> for rf, gr, M0, loc, Δf, b1Map, γ equal the sum of the truncated-pulse
    gradients: every forward family, N = 2 with a dt per entry, nM = 257, nT = 45, s = 7 at K = 16."""
    _, dtype, nC, env, pol, _ = fam
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    p = _problem(31 + nC, 2, 257, 45, nC)
    grads = LEAVES if nC else tuple(k for k in LEAVES if k != 'b1')
    _check_linearity(p, dev, dtype, 7, grads, policy=pol, capfd=capfd, frag='SG=1,REC=1')
    _check_linearity(p, dev, dtype, 7, ('M0', 'rf', 'gr'), policy=pol, capfd=capfd, frag='ROWS=3,SG=0,REC=1')


@pytest.mark.gpu
@pytest.mark.parametrize('case', ['f32-nC1-rf', 'f32-nC1-gr', 'f32-nC2-rf', 'f32-nC2-gr', 'f64-nC4-rf', 'f32-nC1-fixed',
                                  'f64-nC1-fixed', 'f32-nC1-Mt-only', 'f64-nC4-Mt-only', 'f32-nC8-s1', 'f64-nC1-nT1',
                                  'f32-nC1-default-ckpt', 'f32-nC1-strict'])
def test_gradient_variants(dev, capfd, monkeypatch, case):
    """rf-only and gr-only (ROWS 1 / 2), a fixed pulse with M0 / Δf gradients only (ROWS 0), a loss on Mt only, s = 1,
    nT = 1, the default checkpoint interval and 'strict'."""
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    dtype = f64 if case.startswith('f64') else f32
    nC = int(re.search(r'nC(\d+)', case).group(1))
    nT = 1 if 'nT1' in case else 45
    p = _problem(41 + nC, 2, 257, nT, nC)
    kw = dict(capfd=capfd)
    if case.endswith('-rf'):
        grads, kw['frag'] = ('rf',), ('ROWS=1,SG=0,REC=1' if dtype == f32 and nC <= 2 else 'SG=0,REC=1')
    elif case.endswith('-gr'):
        grads, kw['frag'] = ('gr',), ('ROWS=2,SG=0,REC=1' if dtype == f32 and nC <= 2 else 'SG=0,REC=1')
    elif case.endswith('-fixed'):
        grads, kw['frag'] = ('M0', 'df'), 'ROWS=0,SG=1,REC=1'
    elif case.endswith('Mt-only'):
        grads, kw['on_M'] = LEAVES, False
        kw['frag'] = 'SG=1,REC=1'
    else:
        grads = LEAVES
    s = 1 if ('s1' in case or nT == 1) else 7
    if case.endswith('default-ckpt'):
        kw['K'] = None
    if case.endswith('strict'):
        kw['policy'], kw['capfd'] = 'strict', None
    _check_linearity(p, dev, dtype, s, grads, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype,nC', [(f32, 1), (f32, 2), (f32, 8), (f64, 1), (f64, 4)])
def test_ragged_and_multi_tile(dev, capfd, monkeypatch, dtype, nC):
    """One spin past a full tile (257 packed, 129 generic), with dL/dMt only on that last spin: padding lanes must not add
    it a second time.  Then several tiles per CTA (MRPHY_B200_MAX_CTAS=6) on the whole loss."""
    monkeypatch.setenv('MRPHY_B200_DEBUG', '1')
    nM = 257 if (dtype == f32 and nC <= 2) else 129
    p = _problem(51 + nC, 1, nM, 45, nC)
    nT, s = 45, 7
    wt = torch.zeros(1, nM, nT // s, 3, dtype=f64)
    wt[:, -1] = torch.rand(nT // s, 3, generator=torch.Generator().manual_seed(1), dtype=f64) - 0.5
    _, _, g = _run(p, dev, dtype, 16, record=s, grads=LEAVES, wt=wt)
    ref = _linear_reference(p, dev, dtype, 16, s, LEAVES, None, wt)
    tol = 1e-10 if dtype == f64 else 1e-4
    for k in LEAVES:
        assert rel(g[k], ref[k]) <= tol, (k, rel(g[k], ref[k]))
    assert float(g['df'][:, :-1].abs().max()) == 0.0
    monkeypatch.setenv('MRPHY_B200_MAX_CTAS', '6')
    p = _problem(61 + nC, 1, 6 * nM, 45, nC)
    _check_linearity(p, dev, dtype, s, LEAVES, capfd=capfd)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype,nC', [(f32, 1), (f32, 2), (f32, 8), (f64, 4)])
def test_loss_on_M_only_is_unchanged(dev, dtype, nC):
    """record set, loss on M only: M and every gradient bitwise those of the call without record."""
    p = _problem(71 + nC, 2, 257, 45, nC)
    w, _ = _weights(3, 2, 257, 45, 7)
    for grads in (LEAVES, ('M0', 'rf', 'gr')):
        M1, _, g1 = _run(p, dev, dtype, 16, record=7, grads=grads, w=w)
        M0, _, g0 = _run(p, dev, dtype, 16, grads=grads, w=w)
        assert torch.equal(M1, M0)
        for k in grads:
            assert torch.equal(g1[k], g0[k]), k


@pytest.mark.gpu
def test_finite_differences_fp64(dev):
    """Central differences of L = sum_r <w_r, Mt_r> + <w, M> in a few Δf and rf entries (fp64)."""
    p = _problem(81, 1, 20, 40, 1)
    w, wt = _weights(9, 1, 20, 40, 5)
    _, _, g = _run(p, dev, f64, 16, record=5, grads=('rf', 'df'), w=w, wt=wt)

    def loss(q):
        M, Mt, _ = _run(q, dev, f64, 16, record=5)
        return float((M.cpu() * w).sum() + (Mt.cpu() * wt).sum())
    for k, ix, h in (('df', (0, 3), 1e-3), ('df', (0, 17), 1e-3), ('rf', (0, 0, 4, 0), 1e-6), ('rf', (0, 1, 33, 0), 1e-6)):
        qp, qm = dict(p), dict(p)
        qp[k], qm[k] = p[k].clone(), p[k].clone()
        qp[k][ix] += h
        qm[k][ix] -= h
        fd = (loss(qp) - loss(qm)) / (2 * h)
        an = float(g[k].cpu()[ix])
        assert abs(fd - an) <= 1e-5 * abs(an) + 1e-8, (k, ix, fd, an)   # (the loss's rounding / 2h is ~1e-9)


@pytest.mark.gpu
def test_spincube_embed_and_update(dev):
    """SpinCube.applypulse(record=..., doEmbed=True) on a masked cube: NaN outside the mask, the compact values inside;
    doUpdate stores M only."""
    from mrphy import mobjs
    kw = {'dtype': f64, 'device': dev}
    mask = torch.rand(1, 6, 5, 4, generator=torch.Generator().manual_seed(2)) > 0.4
    cube = mobjs.SpinCube((1, 6, 5, 4), tensor([[20., 20., 20.]]), mask=mask, **kw)
    gen = torch.Generator().manual_seed(3)
    pulse = mobjs.Pulse(rf=(torch.rand(1, 2, 30, generator=gen, dtype=f64) * 0.1).to(dev),
                        gr=(torch.rand(1, 3, 30, generator=gen, dtype=f64)).to(dev), **kw)
    M_, Mt_ = cube.applypulse(pulse, record=4)
    M, Mt = cube.applypulse(pulse, record=4, doEmbed=True)
    assert Mt.shape == (1, 6, 5, 4, 7, 3) and M.shape == (1, 6, 5, 4, 3)
    m = mask[0].to(dev)
    assert torch.isnan(Mt[0][~m]).all() and torch.equal(Mt[0][m], Mt_[0])
    assert torch.equal(M[0][m], M_[0])
    M2 = cube.applypulse(pulse)
    assert torch.equal(M2, M_)
    old = cube.M_.clone()
    M3, _ = cube.applypulse(pulse, record=4, doUpdate=True)
    assert torch.equal(cube.M_, M3) and not torch.equal(cube.M_, old)


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [f32, f64])
def test_design_waveform_two_stage(dev, monkeypatch, dtype):
    """rf = tρθ2rf(ρ, θ, rfmax), gr = s2g(ts2s(ts, smax), dt) with record and a loss on Mt and M: the same design-variable
    gradients as with MRPHY_B200_FUSE_DESIGN=0 (1e-12 / 1e-6 relative)."""
    from mrphy import _ops, utils
    N, nM, nT = 2, 301, 133
    gen = torch.Generator().manual_seed(43)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    d = dict(rho=U(N, 1, nT) * 2, theta=U(N, 1, nT) * 3, ts=U(N, 3, nT) * 1.5, rfmax=0.15 + 0.05 * U(N).abs(),
             smax=1.2e4 + 2e3 * U(N, 3).abs(), dt=tensor([4e-6], dtype=f64))
    p = _problem(44, N, nM, nT, 1)
    w, wt = _weights(5, N, nM, nT, 10)
    kw = {'dtype': dtype, 'device': dev}
    out = []
    for fuse in ('1', '0'):
        monkeypatch.setenv('MRPHY_B200_FUSE_DESIGN', fuse)
        v = {k: x.to(**kw) for k, x in d.items()}
        rho, theta, ts = (v[k].requires_grad_(True) for k in ('rho', 'theta', 'ts'))
        rf, gr = utils.tρθ2rf(rho, theta, v['rfmax']), utils.s2g(utils.ts2s(ts, v['smax']), v['dt'])
        t = {k: (None if x is None else x.to(**kw)) for k, x in p.items()}
        M, Mt = _ops.fused_applypulse(t['M0'], rf, gr, t['loc'], Δf_=t['df'], b1Map_=t['b1'], T1_=t['T1'], T2_=t['T2'],
                                      γ_=p['gam'].to(dev), dt=p['dt'].to(dev), record=10)
        ((M * w.to(M)).sum() + (Mt * wt.to(Mt)).sum()).backward()
        out.append((rho.grad, theta.grad, ts.grad))
    for a, b in zip(*out):
        assert rel(a, b) <= (1e-12 if dtype == f64 else 1e-6), rel(a, b)


@pytest.mark.gpu
def test_graph_capture_loss_on_Mt(dev):
    from mrphy import graphs, mobjs
    kw = {'dtype': f32, 'device': dev}
    gen = torch.Generator().manual_seed(4)
    U = lambda *s: (torch.rand(s, generator=gen) * 2 - 1).to(dev)
    sp = mobjs.SpinArray((1, 2000), **kw)
    loc = U(1, 2000, 3) * 5
    df = (U(1, 2000) * 100).requires_grad_(True)
    pulse = mobjs.Pulse(rf=(U(1, 2, 100) * 0.1).requires_grad_(True), gr=(U(1, 3, 100) * 2).requires_grad_(True), **kw)
    step = graphs.capture(lambda: sp.applypulse(pulse, loc_=loc, Δf_=df, record=10)[1][..., 0].pow(2).sum().backward(),
                          params=[df, pulse.rf, pulse.gr])
    step.replay()
    torch.cuda.synchronize()
    first = [df.grad.clone(), pulse.rf.grad.clone(), pulse.gr.grad.clone()]
    d2 = df.detach().clone().requires_grad_(True)
    rf2, gr2 = pulse.rf.detach().clone().requires_grad_(True), pulse.gr.detach().clone().requires_grad_(True)
    p2 = mobjs.Pulse(rf=rf2, gr=gr2, **kw)
    sp.applypulse(p2, loc_=loc, Δf_=d2, record=10)[1][..., 0].pow(2).sum().backward()
    for a, b in zip(first, (d2.grad, rf2.grad, gr2.grad)):
        assert torch.equal(a, b)


@pytest.mark.gpu
def test_scale_memory(dev):
    """128³ spins x 2000 steps, fp32, s = 16: peak memory at most the step without record + Mt + dL/dMt + 256 MB; 256
    seeded spins of Mt agree with the oracle."""
    from mrphy import _ops
    nM, nT, s = 128 ** 3, 2000, 16
    gen = torch.Generator(device=dev).manual_seed(0)
    U = lambda *sh: torch.rand(sh, generator=gen, device=dev) * 2 - 1
    M0 = torch.nn.functional.normalize(U(1, nM, 3), dim=-1)
    loc, df = U(1, nM, 3) * 12, U(1, nM) * 100
    rf, gr = (U(1, 2, nT) * 0.1).requires_grad_(True), (U(1, 3, nT) * 2).requires_grad_(True)
    kw = dict(Δf_=df, γ_=tensor(4257.6, dtype=f64), dt=tensor(4e-6, dtype=f64))
    # weights of the loss on Mt, held in the kernel layout: mul's gradient then comes back in it (no layout copy)
    wt = (torch.rand(1, nT // s, 3, nM, generator=gen, device=dev) - 0.5).permute(0, 3, 1, 2)
    peaks = []
    for record in (None, s):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        out = _ops.fused_applypulse(M0, rf, gr, loc, record=record, **kw)
        if record is None:
            out.sum().backward()
        else:
            (out[0].sum() + (out[1] * wt).sum()).backward()
        torch.cuda.synchronize()
        peaks.append(torch.cuda.max_memory_allocated() - base)
        if record is not None:
            Mt = out[1].detach()
        del out
        rf.grad = gr.grad = None
    mt_bytes = nM * (nT // s) * 3 * 4
    assert peaks[1] <= peaks[0] + 2 * mt_bytes + 256 * 2 ** 20, (peaks, mt_bytes)
    sub = torch.randperm(nM, generator=torch.Generator().manual_seed(3))[:256].to(dev)
    c = lambda x: x.detach()[:, sub].cpu().double()
    q = dict(rf=rf.detach().cpu().float().double(), gr=gr.detach().cpu().float().double(), loc=c(loc), df=c(df), b1=None,
             M0=c(M0), gam=torch.full((1, 256), 4257.6, dtype=f64), dt=tensor(4e-6, dtype=f64), T1=None, T2=None)
    from oracle import bloch_oracle as orc
    ref = _oracle_states(q)[:, :, s - 1::s]
    B = orc.rfgr2beff(q['rf'], q['gr'], q['loc'], q['df'], None, gamma=q['gam'], dtype=f32)
    _, h32 = orc.blochsim_fwd(q['M0'], B, None, None, gamma=q['gam'], dt=q['dt'], dtype=f32, history=True)
    own = float((h32[s::s].permute(1, 2, 0, 3).double() - ref[:, :, :-1]).abs().max())
    err = float((Mt[:, sub].cpu().double() - ref).abs().max())
    assert err <= max(1e-5, 2 * own), (err, own)


# ---------------------------------------------------------------------------------------------------------- host only
def test_record_fields_mirror_matches_library():
    from mrphy import _cabi
    L = _cabi.lib()
    F = _cabi.FusedArgs
    assert L.mrphy_sizeof_args(1) == ctypes.sizeof(F)
    assert (F.every.offset, F.nR.offset) == (F.partials.offset + ctypes.sizeof(ctypes.c_void_p), F.partials.offset + 12)
    assert F.Mt.offset == F.nR.offset + 4 and F.gMt.offset == F.Mt.offset + ctypes.sizeof(ctypes.c_void_p)
    assert L.mrphy_abi_version() == _cabi.ABI_VERSION == 7
    assert {'mrphy_blochsim_fused_fwd', 'mrphy_blochsim_fused_bwd'} <= set(_cabi.EXPORTS)


def _refusable_args():
    """FusedArgs whose checks all pass up to the options; the pointers are never dereferenced: the checks come first."""
    from mrphy import _cabi
    a = _cabi.FusedArgs()
    a.dtype, a.N, a.nM, a.nT, a.nC, a.K = _cabi.MRPHY_F32, 1, 4, 10, 1, 8
    for p in ('Mi', 'rf', 'gr', 'loc', 'Mo', 'ckpt', 'wave', 'gMo', 'partials', 'grf', 'ggr'):
        setattr(a, p, 256)
    a.gamma.ptr = a.dt.ptr = 256
    return a


def test_fused_entry_points_refuse_bad_record_fields():
    """Inconsistent every / nR and null buffers come back as MRPHY_ERR_ARG before anything is launched."""
    from mrphy import _cabi
    L = _cabi.lib()
    for every, nR, mt, gmt, bwd, msg in ((0, 0, 256, 256, False, 'every'), (11, 0, 256, 256, False, 'every'),
                                         (3, 4, 256, 256, False, 'nR'), (3, 3, None, 256, False, 'Mt is null'),
                                         (3, 3, 256, None, True, 'gMt is null'), (2, 4, 256, 256, True, 'nR')):
        a = _refusable_args()
        a.every, a.nR, a.Mt, a.gMt = every, nR, mt, gmt
        rc = L.mrphy_blochsim_fused_bwd(a, 1, None) if bwd else L.mrphy_blochsim_fused_fwd(a, None)
        assert rc == -1, (every, nR, rc)
        assert L.mrphy_last_launch_count() == 0
        err = L.mrphy_last_error().decode()
        assert 'record' in err and (msg in err or 'nR == nT / every' in err), err


@pytest.mark.parametrize('other', ['record', 'gloc', 'gsz', 'gb1'])
def test_design_tail_refuses_record_and_spin_grads(other):
    """The design tail combines with neither record nor per-spin gradients: MRPHY_ERR_ARG, nothing launched."""
    from mrphy import _cabi
    L = _cabi.lib()
    a = _refusable_args()
    d = _cabi.ReparamArgs()
    d.dtype, d.adjoint, d.N, d.nT, d.nC, d.rf_kind = a.dtype, 1, a.N, a.nT, 1, 1
    d.rho = d.theta = d.rfmax = d.grho = d.gtheta = 256      # a design tail that passes its own checks
    a.design = ctypes.addressof(d)
    if other == 'record':
        a.every, a.nR, a.gMt = 5, 2, 256
    else:
        setattr(a, other, 256)
    assert L.mrphy_blochsim_fused_bwd(a, 1, None) == -1
    assert L.mrphy_last_launch_count() == 0
    assert 'design' in L.mrphy_last_error().decode()


@pytest.mark.parametrize('nC', [0, 1, 8])
def test_record_fakes_allocate_implementation_shapes(nC):
    from mrphy import _cabi, _ops
    N, nM, nT, every = 2, 37, 50, 7
    e = lambda *s: torch.empty(s, device='meta')
    rf = e(N, 2, nT, nC) if nC else e(N, 2, nT)
    b1 = e(N, nM, 2, nC) if nC else None
    args = (e(N, nM, 3), rf, e(N, 3, nT), e(N, nM, 3), e(N, nM), b1, None, None, e(1, 1), e(1), 16, 0)
    Mo, Mt, ckpt, wave = _ops._fake_blochsim_fused_fwd(*args, every)
    ref = _ops._fake_blochsim_fused_fwd(*args, 0)
    assert Mo.shape == (N, nM, 3) and Mt.shape == (N, nT // every, 3, nM) and ref[1].shape == (0,)
    assert ckpt.shape == ref[2].shape and wave.shape == ref[3].shape and Mt.dtype == Mo.dtype
    want = (True, True, nC > 0)
    out = _ops._fake_blochsim_fused_bwd(Mo, Mt, Mo, ckpt, wave, rf, e(N, 3, nT), e(N, nM, 3), e(N, nM), b1, None, None,
                                        e(1, 1), e(1), 16, _cabi.FLAG_NEED_GMI, every, *want, *(None,) * 6, 0, 0)
    gMi, flat, gloc, gsz, gb1, *design = out
    assert gMi.shape == (N, nM, 3) and flat.shape == (rf.numel() + N * 3 * nT + _ops.GRAD_TAIL,)
    assert gloc.shape == (N, nM, 3) and gsz.shape == (N, nM)
    assert gb1.shape == ((N, nM, 2, nC) if nC else (0,))
    assert all(g.shape == (0,) for g in design)


@pytest.mark.parametrize('record,match', [(0, 'outside'), (31, 'outside'), (-2, 'outside'), (2.5, 'integer'),
                                          (True, 'integer'), ('4', 'integer'), (4.0, 'integer')])
def test_bad_record_raises_before_anything_runs(record, match):
    """record outside [1, nT] or not an integer: ValueError, before the device is even looked at (CPU tensors here)."""
    from mrphy import _ops
    p = _problem(1, 1, 5, 30, 1)
    with pytest.raises(ValueError, match=match):
        _ops.fused_applypulse(p['M0'], p['rf'], p['gr'], p['loc'], b1Map_=p['b1'], γ_=p['gam'], dt=p['dt'], record=record)


def test_explicit_route_refuses_record():
    """More than 16 coils with a b1Map would take the explicit-Beff route, which does not record: ValueError, with and
    without spin gradients, through fused_applypulse and through SpinArray.applypulse."""
    from mrphy import _ops, mobjs
    p = _problem(2, 1, 5, 30, 17)
    with pytest.raises(ValueError, match='16 transmit coils'):
        _ops.fused_applypulse(p['M0'], p['rf'], p['gr'], p['loc'], b1Map_=p['b1'], γ_=p['gam'], dt=p['dt'], record=3)
    sp = mobjs.SpinArray((1, 5), dtype=f64)
    pulse = mobjs.Pulse(rf=p['rf'], gr=p['gr'], dtype=f64)
    for loc in (p['loc'], p['loc'].clone().requires_grad_(True)):
        with pytest.raises(ValueError, match='16 transmit coils'):
            sp.applypulse(pulse, loc_=loc, b1Map_=p['b1'], record=3)
