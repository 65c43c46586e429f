"""Parity of the CUDA path (through the C ABI) with the reference: golden fixtures generated from the
unmodified reference, the CPU oracle on seeded inputs, and size-independent properties at full size.

Tolerances (BASELINE.json north_star): fp64 |dM| <= 1e-12, fp32 |dM| <= 1e-5 *or* the reference's own
fp32-vs-fp64 distance on the same inputs where that is larger (SURVEY App. B: no fp32 evaluation of
this recurrence, the reference's included, gets below ~2e-5 at nT~1000 with multi-radian steps);
rf/gr gradients <= 1e-4 relative in fp32, <= 1e-9 relative in fp64.
"""
import itertools
import os

import numpy as np
import pytest
import torch_ref
import torch
from torch import tensor

pytestmark = pytest.mark.gpu

f32, f64 = torch.float32, torch.float64
ATOL64, ATOL32, RTOL_G32, RTOL_G64 = 1e-12, 1e-5, 1e-4, 1e-9


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available(), 'run with -m gpu on a CUDA box'
    import mrphy  # noqa: F401
    from mrphy import _cabi
    _cabi.lib()
    return torch.device('cuda:0')


def mx(a, b):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    return float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max())


def rel(a, b):
    a = a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    b = b.detach().cpu().numpy() if isinstance(b, torch.Tensor) else np.asarray(b)
    a, b = a.astype(np.float64).ravel(), b.astype(np.float64).ravel()
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


def _fp32_bound(ref32, ref64):
    """The documented fp32 rule (SURVEY 8c, north_star): 1e-5, or the reference algorithm's OWN fp32-vs-fp64 distance on
    the same inputs where that is larger (oracle run in fp32: same operations in the same order as sims.py)."""
    return max(ATOL32, mx(ref32, ref64))


def T(x, dev, dtype):
    return None if x is None else tensor(np.asarray(x), device=dev, dtype=dtype)


def run_fused(g, dev, dtype, w, prefix='in_', names=None, **kw):
    """fixture dict -> (Mo, gM0, grf, ggr) through mrphy._ops.fused_applypulse."""
    from mrphy import _ops
    nm = names or dict(M0='M0', rf='rf', gr='gr', loc='loc', df='df', b1='b1', T1='T1', T2='T2', gam='gam', dt='dt')
    get = lambda k: g.get(prefix + nm[k])
    M0 = T(get('M0'), dev, dtype).requires_grad_(True)
    rf = T(get('rf'), dev, dtype).requires_grad_(True)
    gr = T(get('gr'), dev, dtype).requires_grad_(True)
    Mo = _ops.fused_applypulse(M0, rf, gr, T(get('loc'), dev, dtype), Δf_=T(get('df'), dev, dtype),
                               b1Map_=T(get('b1'), dev, dtype), T1_=T(get('T1'), dev, dtype),
                               T2_=T(get('T2'), dev, dtype), γ_=T(get('gam'), dev, f64), dt=T(get('dt'), dev, f64), **kw)
    (Mo * T(w, dev, dtype)).sum().backward()
    return Mo.detach(), M0.grad, rf.grad, gr.grad


KAT = dict(M0='M0', rf='rf', gr='gr', loc='loc', df='df', b1='b1', T1='T1', T2='T2', gam='gamma', dt='dt')


def test_kat3_golden_constants(dev, golden):
    """tests/test_slowsims.py:77-80 (upstream atol 1e-9)."""
    g = golden('kat3')
    Mo, gM0, grf, ggr = run_fused(g, dev, f64, np.ones((1, 3, 3)), prefix='', names=KAT)
    assert mx(Mo, g['Mo_const']) < ATOL64
    assert rel(grf, g['grf']) < RTOL_G64 and rel(ggr, g['ggr']) < RTOL_G64 and mx(gM0, g['gM0']) < 1e-10
    Mo32, _, grf32, ggr32 = run_fused(g, dev, f32, np.ones((1, 3, 3)), prefix='', names=KAT)
    assert mx(Mo32, g['Mo_const']) < 1e-4          # upstream's own fp32 tolerance (tests/test_sims.py:15)
    assert rel(grf32, g['grf']) < RTOL_G32 and rel(ggr32, g['ggr']) < RTOL_G32


@pytest.mark.parametrize('tag', ['relax', 'norelax'])
def test_sims512_explicit_beff(dev, golden, tag):
    """tests/test_sims.py:104-105,142-143: sims.blochsim grads wrt M0 and Beff (upstream atol 1e-9)."""
    from mrphy import sims, beffective
    g = golden('sims512')
    gam, dt = T(g['gamma'], dev, f64), T(g['dt'], dev, f64)
    M0 = T(g['M0'], dev, f64).requires_grad_(True)
    beff = beffective.rfgr2beff(T(g['rf'], dev, f64), T(g['gr'], dev, f64), T(g['loc'], dev, f64),
                                Δf=T(g['df'], dev, f64), b1Map=T(g['b1'], dev, f64), γ=gam).requires_grad_(True)
    T1, T2 = (T(g['T1'], dev, f64), T(g['T2'], dev, f64)) if tag == 'relax' else (None, None)
    Mo = sims.blochsim(M0, beff, T1=T1, T2=T2, γ=gam, dt=dt)
    Mo.sum().backward()
    assert mx(Mo, g[f'Mo_{tag}']) < ATOL64
    assert mx(M0.grad, g[f'gM0_{tag}']) < 1e-9
    assert mx(beff.grad[:, ::int(g['sub_step'])], g[f'gBeff_sub_{tag}']) < 1e-9
    # the fused path on the same problem returns the waveform gradients of the reference chain
    gg = dict(g, b1=np.broadcast_to(g['b1'], (1, 512, 2, 1)))
    if tag == 'norelax':
        gg.pop('T1'), gg.pop('T2')
    Mo_f, gM0_f, grf, ggr = run_fused(gg, dev, f64, np.ones((1, 512, 3)), prefix='', names=KAT)
    assert mx(Mo_f, g[f'Mo_{tag}']) < ATOL64 and mx(gM0_f, g[f'gM0_{tag}']) < 1e-9
    assert rel(grf, g[f'grf_{tag}']) < RTOL_G64 and rel(ggr, g[f'ggr_{tag}']) < RTOL_G64


def test_cube27_applypulse_goldens(dev, golden):
    """tests/test_mobjs.py:98-131: SpinCube.applypulse through mask/embed; Mo0a (relax) and Mo0b (no relax,
    doUpdate)."""
    from mrphy import mobjs, γH, dt0, _slice
    g = golden('cube27')
    kw = {'dtype': f64, 'device': dev}
    p = mobjs.Pulse(rf=T(g['rf'], dev, f64), gr=T(g['gr'], dev, f64), dt=dt0, **kw)
    mask = tensor(g['mask'], device=dev)
    cube = mobjs.SpinCube((1, 3, 3, 3), T(g['fov'], dev, f64), mask=mask, T1_=tensor([[1.]]), γ=γH, **kw)
    cube.ofst = T(g['ofst'], dev, f64)
    cube.M_ = tensor([0., 1., 0.])
    cube.T2 = tensor([[4e-2]]).expand(cube.shape)
    cube.M_[cube.crds_([_slice, [0, 1], [1, 0], _slice, _slice])] = tensor([1., 0., 0.], **kw)
    cube.M_[cube.crds_([_slice, [2, 1], [1, 2], _slice, _slice])] = tensor([0., 0., 1.], **kw)
    cube.Δf = torch.sum(-cube.loc[0:1, :, :, :, 0:2], dim=-1) * cube.γ
    Ma = cube.applypulse(p, doEmbed=True)
    cube.applypulse(p, doEmbed=True, doRelax=False, doUpdate=True)
    Mb = cube.M
    for M, ref in ((Ma, g['Mo0a']), (Mb, g['Mo0b'])):
        assert M[0:1, 1, :, 1, :].cpu().numpy() == pytest.approx(ref, abs=1e-9)
        assert M[0:1, :, 1, 1, :].cpu().numpy() == pytest.approx(ref, abs=1e-9)
    assert np.allclose(Mb.cpu().numpy(), g['M_norelax'], atol=1e-9, equal_nan=True)
    assert torch.isnan(Ma[0, 0, 0, 0]).all()


@pytest.mark.parametrize('name', ['rand_mc', 'rand_nob1', 'rand_norelax', 'bench8'])
def test_random_fixtures_fp64_and_fp32(dev, golden, name):
    """Multi-coil + per-spin constants, summed coils + per-batch dt, no relaxation, bench distributions."""
    g = golden(name)
    w = g['in_w'] if 'in_w' in g else 2 * (g['Mo_f64'] - np.array([0., 1., 0.]))
    Mo, gM0, grf, ggr = run_fused(g, dev, f64, w)
    assert mx(Mo, g['Mo_f64']) < ATOL64
    assert rel(grf, g['grf_f64']) < RTOL_G64 and rel(ggr, g['ggr_f64']) < RTOL_G64
    if 'gM0_slow_f64' in g:
        assert rel(gM0, g['gM0_slow_f64']) < RTOL_G64
    floor = mx(g['Mo_f32'], g['Mo_f64'])            # the reference's own fp32 error on these inputs
    if 'grf_f32' in g:
        print(f'[{name}/reference fp32] grf rel={rel(g["grf_f32"], g["grf_f64"]):.2e} ggr rel={rel(g["ggr_f32"], g["ggr_f64"]):.2e}')
    for trig in ('fast', 'mixed', 'precise'):
        from mrphy import _cabi
        fl = {'precise': _cabi.FLAG_TRIG_PRECISE, 'mixed': _cabi.FLAG_TRIG_PRECISE | _cabi.FLAG_TRIG_FAST_BWD, 'fast': 0}[trig]
        Mo32, _, grf32, ggr32 = run_fused(g, dev, f32, w, flags=fl)
        d = mx(Mo32, g['Mo_f64'])
        print(f'[{name}/{trig}] fp32 max|dM|={d:.2e} (reference fp32: {floor:.2e}) '
              f'grf rel={rel(grf32, g["grf_f64"]):.2e} ggr rel={rel(ggr32, g["ggr_f64"]):.2e}')
        # default policy ('precise') must not be worse than the reference's own fp32; raw MUFU trig may be 2.5x
        assert d < max(ATOL32, (2.5 if trig == 'fast' else 1.0) * floor)
        assert rel(grf32, g['grf_f64']) < RTOL_G32 and rel(ggr32, g['ggr_f64']) < RTOL_G32


def _random_problem(seed, N, nM, nT, nC, has_b1, relax, dtype=f64):
    gen = torch.Generator().manual_seed(seed)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    p = dict(rf=U(N, 2, nT, nC) * 0.1 if nC else U(N, 2, nT) * 0.1, gr=U(N, 3, nT) * 2, loc=U(N, nM, 3) * 12,
             df=U(N, nM) * 200, b1=None, M0=torch.nn.functional.normalize(U(N, nM, 3), dim=-1),
             gam=tensor(4257.6, dtype=f64) * (1 + 0.02 * U(N, nM)), dt=tensor([4e-6], dtype=f64),
             T1=(1.0 + 0.5 * U(N, nM)) if relax else None, T2=(0.06 + 0.05 * U(N, nM)) if relax else None,
             w=U(N, nM, 3))
    if has_b1:
        b1 = U(N, nM, 2, max(nC, 1)) * 0.1
        b1[:, :, 0] += 1
        p['b1'] = b1
    return {k: (None if v is None else v.to(dtype).to(f64)) for k, v in p.items()}


@pytest.mark.parametrize('K', [1, 7, 16, 64])
@pytest.mark.parametrize('shape', [(1, 130, 75, 1), (2, 300, 333, 2), (1, 1, 1, 0), (3, 129, 64, 4), (1, 200, 70, 8),
                                   (2, 131, 33, 16), (1, 150, 41, 3)])
def test_fused_vs_oracle_ragged(dev, K, shape):
    """Ragged sizes (nM not a multiple of the CTA, nT not a multiple of K), nCoils 1/2/3/4/8/16 (8 and 16: step-major staged
    waveform; all multi-coil: weights applied in the reduce phase), N>1."""
    from oracle import bloch_oracle as orc
    N, nM, nT, nC = shape
    p = _random_problem(10 + nM, N, nM, nT, nC, has_b1=nC > 0, relax=True)
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'],
                                 T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    g = {('in_' + k): (None if v is None else v.numpy()) for k, v in p.items()}
    g = {k: v for k, v in g.items() if v is not None}
    Mo, gM0, grf, ggr = run_fused(g, dev, f64, p['w'].numpy(), ckpt=K)
    assert mx(Mo, ref['Mo']) < ATOL64
    assert rel(grf, ref['grf']) < RTOL_G64 and rel(ggr, ref['ggr']) < RTOL_G64 and rel(gM0, ref['gM0']) < RTOL_G64
    Mo32, gM032, grf32, ggr32 = run_fused(g, dev, f32, p['w'].numpy(), ckpt=K)
    p32 = {k: (None if v is None else v.to(f32)) for k, v in p.items()}      # the reference algorithm in fp32, same inputs
    ref32 = orc.applypulse_fwd_bwd(p32['M0'], p32['rf'], p32['gr'], p32['loc'], p32['w'], df=p32['df'], b1=p32['b1'],
                                   T1=p32['T1'], T2=p32['T2'], gamma=p32['gam'], dt=p32['dt'], dtype=f32)
    assert mx(Mo32, ref['Mo']) < _fp32_bound(ref32['Mo'], ref['Mo']), (mx(Mo32, ref['Mo']), mx(ref32['Mo'], ref['Mo']))
    assert rel(grf32, ref['grf']) < RTOL_G32 and rel(ggr32, ref['ggr']) < RTOL_G32


@pytest.mark.parametrize('nC', [3, 4, 8, 16])
def test_tensor_core_transmit_field_matches_fma_path_and_oracle(dev, nC, monkeypatch):
    """fp32 forward with >= 3 coils: the transmit field sum_c b1_c rf_c comes from tcgen05.mma (TF32 operands split in two
    exactly representable parts, fused_fwd_tc_kernel) instead of 4 nCoils FMAs per spin and step.  Must (1) be taken
    (debug line of the launcher), (2) agree with the FMA kernels (MRPHY_B200_TC=0) to fp32 rounding, (3) track the fp64 oracle
    as well as the reference algorithm in fp32, (4) leave the gradients -- whose backward re-stages the waveform in its own
    layout over the tensor-core operand tiles -- unchanged, (5) step aside for checkpoint intervals above 32 steps.
    Three tiles of spins, ragged in spins and steps (nT = 203: 7 chunks, the last of 11 steps)."""
    from oracle import bloch_oracle as orc
    p = _random_problem(300 + nC, 2, 300, 203, nC, has_b1=True, relax=True, dtype=f32)
    g = {('in_' + k): v.numpy() for k, v in p.items()}
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'], T2=p['T2'],
                                 gamma=p['gam'], dt=p['dt'])
    p32 = {k: v.to(f32) for k, v in p.items()}
    ref32 = orc.applypulse_fwd_bwd(p32['M0'], p32['rf'], p32['gr'], p32['loc'], p32['w'], df=p32['df'], b1=p32['b1'],
                                   T1=p32['T1'], T2=p32['T2'], gamma=p32['gam'], dt=p32['dt'], dtype=f32)
    monkeypatch.setenv('MRPHY_B200_TC', '0')
    Mo_fma, gM_fma, grf_fma, ggr_fma = run_fused(g, dev, f32, p['w'].numpy(), ckpt=32)
    monkeypatch.setenv('MRPHY_B200_TC', '1')
    Mo_tc, gM_tc, grf_tc, ggr_tc = run_fused(g, dev, f32, p['w'].numpy(), ckpt=32)
    d_paths, d_tc, d_fma, floor = mx(Mo_tc, Mo_fma), mx(Mo_tc, ref['Mo']), mx(Mo_fma, ref['Mo']), mx(ref32['Mo'], ref['Mo'])
    print(f'[tensor-core field nC={nC}] |M_tc - M_fma| {d_paths:.2e}; vs fp64 oracle: tc {d_tc:.2e}, fma {d_fma:.2e}, '
          f'reference algorithm in fp32 {floor:.2e}')
    assert not torch.equal(Mo_tc, Mo_fma), 'tensor-core path not taken'      # different rounding order: never bit-identical
    assert d_paths < 6e-6                                                     # each is ~4.5e-6 from the fp64 oracle
    assert d_tc < _fp32_bound(ref32['Mo'], ref['Mo'])
    assert rel(grf_tc, ref['grf']) < RTOL_G32 and rel(ggr_tc, ref['ggr']) < RTOL_G32 and rel(gM_tc, ref['gM0']) < RTOL_G32
    assert rel(grf_tc, grf_fma) < 2e-5 and rel(ggr_tc, ggr_fma) < 2e-5
    # K = 64 > 32: the FMA kernels run whatever the switch says -> bit-identical to MRPHY_B200_TC=0
    Mo64, _, _, _ = run_fused(g, dev, f32, p['w'].numpy(), ckpt=64)
    monkeypatch.setenv('MRPHY_B200_TC', '0')
    Mo64_fma, _, _, _ = run_fused(g, dev, f32, p['w'].numpy(), ckpt=64)
    assert torch.equal(Mo64, Mo64_fma)


@pytest.mark.parametrize('shape', [(1, 1, 1, 4), (2, 5, 3, 8), (1, 127, 9, 16), (70, 3, 40, 4)])
def test_tensor_core_forward_tiny_and_many_entries(dev, shape):
    """Edge sizes of the tensor-core forward: a single spin and a single step (one TMEM lane, 2 of 16 operand rows live), fewer
    spins than one tile, more batch entries than resident CTA slots per entry (N = 70)."""
    from oracle import bloch_oracle as orc
    N, nM, nT, nC = shape
    p = _random_problem(500 + nM, N, nM, nT, nC, has_b1=True, relax=True, dtype=f32)
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'], T2=p['T2'],
                                 gamma=p['gam'], dt=p['dt'])
    g = {('in_' + k): v.numpy() for k, v in p.items()}
    Mo, gM0, grf, ggr = run_fused(g, dev, f32, p['w'].numpy())
    assert mx(Mo, ref['Mo']) < ATOL32
    assert rel(grf, ref['grf']) < RTOL_G32 and rel(ggr, ref['ggr']) < RTOL_G32 and rel(gM0, ref['gM0']) < RTOL_G32


def test_tensor_core_forward_is_graph_capturable_and_batched(dev):
    """The tensor-core forward inside a captured design step (its launcher queries function attributes, sets the dynamic
    shared-memory limit and allocates TMEM in-kernel: none of it may break stream capture), with N = 3 batch entries of
    different pulses: replays reproduce the eager gradients bit for bit."""
    from mrphy import _ops, graphs
    p = _random_problem(411, 3, 260, 96, 8, has_b1=True, relax=True, dtype=f32)
    q = {k: T(v.numpy(), dev, f32) for k, v in p.items()}
    gam, dts = T(p['gam'].numpy(), dev, f64), T(p['dt'].numpy(), dev, f64)
    rf, gr = q['rf'].clone().requires_grad_(True), q['gr'].clone().requires_grad_(True)

    def step():
        Mo = _ops.fused_applypulse(q['M0'], rf, gr, q['loc'], Δf_=q['df'], b1Map_=q['b1'], T1_=q['T1'], T2_=q['T2'], γ_=gam, dt=dts)
        (Mo * q['w']).sum().backward()

    step()
    want = (rf.grad.clone(), gr.grad.clone())
    assert float(want[0].abs().max()) > 0
    captured = graphs.capture(step, params=(rf, gr))
    for _ in range(2):
        captured.replay()
        torch.cuda.synchronize()
        assert torch.equal(rf.grad, want[0]) and torch.equal(gr.grad, want[1])


@pytest.mark.parametrize('K', [100, 128])
def test_single_coil_fp32_chunks_up_to_128_steps(dev, K):
    """The fp32 single-coil kernels stage up to 128 steps per chunk (checkpoint interval K <= 128; the default picks 128 when the
    relaxation allows it); every other kernel family stops at 64 and says so."""
    from oracle import bloch_oracle as orc
    from mrphy import _ops
    p = _random_problem(700 + K, 2, 300, 333, 1, has_b1=True, relax=True, dtype=f32)
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'], T2=p['T2'],
                                 gamma=p['gam'], dt=p['dt'])
    p32 = {k: v.to(f32) for k, v in p.items()}
    ref32 = orc.applypulse_fwd_bwd(p32['M0'], p32['rf'], p32['gr'], p32['loc'], p32['w'], df=p32['df'], b1=p32['b1'],
                                   T1=p32['T1'], T2=p32['T2'], gamma=p32['gam'], dt=p32['dt'], dtype=f32)
    g = {('in_' + k): v.numpy() for k, v in p.items()}
    Mo, gM0, grf, ggr = run_fused(g, dev, f32, p['w'].numpy(), ckpt=K)
    assert mx(Mo, ref['Mo']) < _fp32_bound(ref32['Mo'], ref['Mo'])
    assert rel(grf, ref['grf']) < RTOL_G32 and rel(ggr, ref['ggr']) < RTOL_G32 and rel(gM0, ref['gM0']) < RTOL_G32
    Mo64, _, grf64, _ = run_fused(g, dev, f32, p['w'].numpy(), ckpt=64)
    assert torch.equal(Mo, Mo64) and rel(grf, grf64) < 1e-5          # the forward does not depend on K, the adjoint barely
    assert _ops.pick_ckpt_interval(T(p['dt'].numpy(), dev, f64), None, None, _ops.K_MAX1) == 128
    with pytest.raises(RuntimeError, match='checkpoint interval'):
        run_fused(g, dev, f64, p['w'].numpy(), ckpt=K)               # fp64: 64 at most


def test_batch_sharding_needs_no_collective(dev):
    """mrphy.parallel.shard_batch: the batch axis as the shard axis (SURVEY 8e).  Both "ranks" of a world of 2, run one after the
    other on this GPU, together reproduce the unsharded magnetisation and -- through the views of the caller's leaves -- its
    rf / gr gradients bit for bit, with no all-reduce."""
    from mrphy import mobjs, parallel
    kw = {'dtype': f32, 'device': dev}
    gen = torch.Generator().manual_seed(12)
    N, n, nT = 4, 6, 50
    cube = mobjs.SpinCube((N, n, n, n), tensor([[24., 24., 24.]]), **kw)
    cube.Δf = (torch.rand(N, n, n, n, generator=gen) * 200 - 100).to(dev)
    b1 = (torch.rand(N, n ** 3, 2, generator=gen) * 0.2 + tensor([0.9, -0.1])).to(dev)
    rf0, gr0 = (torch.rand(N, 2, nT, generator=gen) * 0.2 - 0.1).to(dev), (torch.rand(N, 3, nT, generator=gen) * 4 - 2).to(dev)
    w = (torch.rand(N, n ** 3, 3, generator=gen) * 2 - 1).to(dev)
    pulse = mobjs.Pulse(rf=rf0.clone().requires_grad_(True), gr=gr0.clone().requires_grad_(True), **kw)
    M = cube.applypulse(pulse, b1Map_=b1)
    (M * w).sum().backward()
    want = (M.detach().clone(), pulse.rf.grad.clone(), pulse.gr.grad.clone())
    pulse2 = mobjs.Pulse(rf=rf0.clone().requires_grad_(True), gr=gr0.clone().requires_grad_(True), **kw)
    outs = []
    for rank in range(2):
        sp, kws, pl, (lo, hi) = parallel.shard_batch(cube, pulse2, rank, 2, b1Map_=b1)
        Ml = sp.applypulse(pl, **kws)
        (Ml * w[lo:hi]).sum().backward()
        outs.append(Ml.detach())
    assert torch.equal(torch.cat(outs), want[0])
    assert torch.equal(pulse2.rf.grad, want[1]) and torch.equal(pulse2.gr.grad, want[2])


def test_multi_tile_ctas_accumulate(dev, monkeypatch):
    """Force a 3-CTA grid so every CTA walks several spin tiles (partial-sum read-modify-write path)."""
    from oracle import bloch_oracle as orc
    p = _random_problem(77, 2, 1500, 96, 1, has_b1=True, relax=True)
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'],
                                 T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    g = {('in_' + k): v.numpy() for k, v in p.items() if v is not None}
    monkeypatch.setenv('MRPHY_B200_MAX_CTAS', '6')
    Mo, gM0, grf, ggr = run_fused(g, dev, f64, p['w'].numpy())
    assert mx(Mo, ref['Mo']) < ATOL64 and rel(grf, ref['grf']) < RTOL_G64 and rel(ggr, ref['ggr']) < RTOL_G64
    assert rel(gM0, ref['gM0']) < RTOL_G64


def test_cta_cap_below_sm_aware_grid(dev, monkeypatch):
    """MRPHY_B200_MAX_CTAS below the SM-aware backward grid (one batch entry, >= 2 tiles per SM): the grid must stay
    inside the partial-sum workspace that was sized from the cap (ADVICE r1: out-of-bounds partial sums otherwise)."""
    from oracle import bloch_oracle as orc
    p = _random_problem(78, 1, 80000, 24, 1, has_b1=True, relax=True, dtype=f32)
    g = {('in_' + k): v.numpy() for k, v in p.items() if v is not None}
    a = run_fused(g, dev, f32, p['w'].numpy())
    monkeypatch.setenv('MRPHY_B200_MAX_CTAS', '200')
    b = run_fused(g, dev, f32, p['w'].numpy())
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    assert rel(b[2], a[2]) < 1e-5 and rel(b[3], a[3]) < 1e-5        # another partition of the spin sum: rounding only
    sub = slice(0, 64)
    ref = orc.applypulse_fwd_bwd(p['M0'][:, sub], p['rf'], p['gr'], p['loc'][:, sub], p['w'][:, sub], df=p['df'][:, sub],
                                 b1=p['b1'][:, sub], T1=p['T1'][:, sub], T2=p['T2'][:, sub], gamma=p['gam'][:, sub], dt=p['dt'])
    assert mx(b[0][:, sub], ref['Mo']) < ATOL32 and rel(b[1][:, sub], ref['gM0']) < RTOL_G32


def test_explicit_beff_vs_oracle_and_fused(dev):
    from oracle import bloch_oracle as orc
    from mrphy import sims, beffective
    p = _random_problem(5, 2, 200, 150, 1, has_b1=True, relax=True)
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'],
                                 T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    p32 = {k: (None if v is None else v.to(f32)) for k, v in p.items()}
    ref32 = orc.applypulse_fwd_bwd(p32['M0'], p32['rf'], p32['gr'], p32['loc'], p32['w'], df=p32['df'], b1=p32['b1'],
                                   T1=p32['T1'], T2=p32['T2'], gamma=p32['gam'], dt=p32['dt'], dtype=f32)
    for dtype, tolM, tolG in ((f64, ATOL64, RTOL_G64), (f32, _fp32_bound(ref32['Mo'], ref['Mo']), RTOL_G32)):
        c = lambda k: None if p[k] is None else p[k].to(dev, dtype)
        rf, gr = c('rf').requires_grad_(True), c('gr').requires_grad_(True)
        M0 = c('M0').requires_grad_(True)
        beff = beffective.rfgr2beff(rf, gr, c('loc'), Δf=c('df'), b1Map=c('b1'), γ=c('gam'))
        beff.retain_grad()
        # (N,*Nd) with Nd=(20,10): exercises the flattening of per-spin constants
        Nd = (20, 10)
        Mo = sims.blochsim(M0.reshape(2, *Nd, 3), beff.reshape(2, *Nd, 150, 3), T1=c('T1').reshape(2, *Nd),
                           T2=c('T2').reshape(2, *Nd), γ=c('gam').reshape(2, *Nd), dt=c('dt'))
        assert Mo.shape == (2, 20, 10, 3) and Mo.dtype == dtype
        (Mo.reshape(2, 200, 3) * c('w')).sum().backward()
        assert mx(Mo.reshape(2, 200, 3), ref['Mo']) < tolM
        assert rel(beff.grad, ref['gBeff']) < tolG and rel(M0.grad, ref['gM0']) < tolG
        assert rel(rf.grad, ref['grf']) < tolG and rel(gr.grad, ref['ggr']) < tolG


@pytest.mark.parametrize('dtype,nM,nT,case', [
    # 16-byte-aligned rows (nT % 4 == 0 in fp32, even in fp64): 16-byte copies
    (f32, 200, 152, ''), (f32, 64, 16, ''), (f32, 1, 4, ''), (f32, 333, 1000, ''), (f64, 77, 152, ''), (f64, 1, 2, ''),
    # other rows: element copies, and a last tile that ends in a partial group of steps
    (f32, 200, 151, ''), (f32, 45, 17, ''), (f32, 33, 3, ''), (f32, 1, 1, ''), (f64, 77, 151, ''), (f64, 5, 9, ''),
    (f64, 1, 1, ''),
    (f32, 100, 152, 'offset'),                    # aligned nT, but the data pointer is one element into a buffer
    (f32, 70, 151, 'ckpt3'), (f64, 70, 151, 'ckpt3'),   # checkpoints every 3 steps: some inside the partial group
    (f32, 50, 151, 'M0only'),                     # no dL/dBeff is stored
])
def test_explicit_beff_tile_pipeline(dev, monkeypatch, dtype, nM, nT, case):
    """Explicit-field kernels on both row alignments: ragged spin counts (odd, < 32, not a multiple of the CTA), partial
    last tiles and groups, checkpoints that fall inside tiles and groups; values and both gradients against the fp64
    oracle (fp64: 1e-12 / 1e-9; fp32: the fp32 rule)."""
    from oracle import bloch_oracle as orc
    from mrphy import sims
    if case == 'ckpt3':
        monkeypatch.setenv('MRPHY_B200_CKPT', '3')
    p = _random_problem(100 + nM, 2, nM, nT, 1, has_b1=True, relax=True, dtype=dtype)
    beff = orc.rfgr2beff(p['rf'], p['gr'], p['loc'], df=p['df'], b1=p['b1'], gamma=p['gam']).to(dtype)
    Mo64, gM64, gB64 = orc.blochsim_adj(p['M0'], beff, p['w'], T1=p['T1'], T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    if dtype == f32:
        Mo32, _, _ = orc.blochsim_adj(p['M0'].to(f32), beff, p['w'].to(f32), T1=p['T1'].to(f32), T2=p['T2'].to(f32),
                                      gamma=p['gam'].to(f32), dt=p['dt'].to(f32), dtype=f32)
        tolM, tolG = _fp32_bound(Mo32, Mo64), RTOL_G32
    else:
        tolM, tolG = ATOL64, RTOL_G64
    M0 = p['M0'].to(dev, dtype).requires_grad_(True)
    off = 1 if case == 'offset' else 0
    B = torch.empty(beff.numel() + off, dtype=dtype, device=dev)[off:].view(beff.shape)
    B.copy_(beff)
    B.requires_grad_(case != 'M0only')
    es = B.element_size()
    aligned = B.data_ptr() % 16 == 0 and (B.stride(1) * es) % 16 == 0 and (B.stride(0) * es) % 16 == 0
    assert aligned == ((nT * 3 * es) % 16 == 0 and off == 0)     # the case runs the instantiation it was written for
    Mo = sims.blochsim(M0, B, T1=p['T1'].to(dev, dtype), T2=p['T2'].to(dev, dtype), γ=p['gam'].to(dev), dt=p['dt'].to(dev))
    (Mo * p['w'].to(dev, dtype)).sum().backward()
    assert mx(Mo, Mo64) < tolM and rel(M0.grad, gM64) < tolG
    if case == 'M0only':
        assert B.grad is None
    else:
        assert rel(B.grad, gB64) < tolG


def test_defaults_fp64_constants_with_fp32_state(dev):
    """sims.blochsim(Mi32, Beff32) with the float64 0-dim defaults γH, dt0 (SURVEY 8b: output stays fp32)."""
    from mrphy import sims
    from oracle import bloch_oracle as orc
    gen = torch.Generator().manual_seed(3)
    Mi = torch.nn.functional.normalize(torch.rand(1, 50, 3, generator=gen) - .5, dim=-1)
    Beff = (torch.rand(1, 50, 40, 3, generator=gen) - .5) * 2
    Mo = sims.blochsim(Mi.to(dev), Beff.to(dev))
    assert Mo.dtype == f32 and Mo.shape == (1, 50, 3)
    assert mx(Mo, orc.blochsim_fwd(Mi, Beff)) < 5e-6
    # non-contiguous Beff is accepted (upstream accepts it too)
    Bt = Beff.transpose(1, 2).contiguous().transpose(1, 2).to(dev)
    assert mx(sims.blochsim(Mi.to(dev), Bt), Mo) == 0.0


def test_zero_field_is_identity_and_nograd_path(dev):
    from mrphy import _ops
    M0 = torch.nn.functional.normalize(torch.rand(1, 10, 3, dtype=f64, device=dev), dim=-1)
    z = lambda *s: torch.zeros(*s, dtype=f64, device=dev)
    Mo = _ops.fused_applypulse(M0, z(1, 2, 20), z(1, 3, 20), z(1, 10, 3), γ_=tensor(4257.6, device=dev), dt=tensor(4e-6, device=dev))
    assert torch.equal(Mo, M0) and not Mo.requires_grad


def test_doupdate_chain_and_second_backward(dev):
    """Two pulses chained through doUpdate (Mi carries a graph; upstream breaks here, sims.py:267), and
    backward twice with retain_graph (upstream raises: it mutates its saved tensors)."""
    from mrphy import mobjs
    from oracle import bloch_oracle as orc
    kw = {'dtype': f64, 'device': dev}
    gen = torch.Generator().manual_seed(9)
    rf = ((torch.rand(1, 2, 60, generator=gen, dtype=f64) - .5) * .2).to(dev).requires_grad_(True)
    gr = ((torch.rand(1, 3, 60, generator=gen, dtype=f64) - .5) * 4).to(dev).requires_grad_(True)
    cube = mobjs.SpinCube((1, 4, 4, 4), tensor([[24., 24., 24.]]), **kw)
    cube.Δf_ = ((torch.rand(1, 64, generator=gen, dtype=f64) - .5) * 400).to(dev)
    p = mobjs.Pulse(rf=rf, gr=gr, **kw)
    cube.applypulse(p, doUpdate=True)
    M2 = cube.applypulse(p, doUpdate=True)
    assert cube.M_.requires_grad
    loss = (M2[..., 1] ** 2).sum()
    loss.backward(retain_graph=True)
    g1 = rf.grad.clone()
    rf.grad = None
    loss.backward()
    assert torch.equal(g1, rf.grad)
    # oracle: the same two pulses back to back == one pulse of 120 steps
    rr, gg = torch.cat([rf, rf], 2).detach().cpu(), torch.cat([gr, gr], 2).detach().cpu()
    M0 = tensor([0., 0., 1.], dtype=f64).expand(1, 64, 3)
    kwo = dict(df=cube.Δf_.cpu(), T1=1.47, T2=0.07)
    Mo = orc.blochsim_fwd(M0, orc.rfgr2beff(rr, gg, cube.loc_.cpu(), df=cube.Δf_.cpu()), 1.47, 0.07)
    gMo = torch.zeros_like(Mo)
    gMo[..., 1] = 2 * Mo[..., 1]
    ref = orc.applypulse_fwd_bwd(M0, rr, gg, cube.loc_.cpu(), gMo, **kwo)
    assert mx(M2, ref['Mo']) < ATOL64
    assert rel(g1, ref['grf'][:, :, :60] + ref['grf'][:, :, 60:]) < RTOL_G64


def test_bitwise_reproducible_gradients(dev):
    """The spin reduction is atomics-free: two runs give identical bits."""
    p = _random_problem(21, 1, 4096, 128, 1, has_b1=True, relax=True)
    g = {('in_' + k): v.numpy() for k, v in p.items() if v is not None}
    a = run_fused(g, dev, f32, p['w'].numpy())
    b = run_fused(g, dev, f32, p['w'].numpy())
    assert all(torch.equal(x, y) for x, y in zip(a, b))


FULL = {'c2': (1, 64, 1000), 'c3': (1, 128, 2000), 'c4': (64, 40, 1000), 'c5': (1, 256, 4000)}   # BASELINE.json configs


@pytest.mark.parametrize('cfg', ['c2', 'c3', 'c4', 'c5'])
@pytest.mark.parametrize('dtype', [f32, f64])
def test_full_size_properties(dev, dtype, cfg):
    """Every BASELINE config at FULL size -- C2 64^3 x 1000, C3 128^3 x 2000, C4 64 pulses x 40^3 x 1000, C5 256^3 x 4000
    (63 checkpoint segments, a 12.7-GB checkpoint buffer) -- through properties that do not need the reference at these
    sizes (it would need 13.6 GB ... 3.5 TB):
    (1) a random subset of spins (of three batch entries at C4) matches the oracle; fp32 within max(1e-5, the oracle's own
        fp32 error on that subset) for the default policy 'precise' (and 'mixed': same forward), 1e-5 flat for 'strict';
    (2) without relaxation |M| is preserved;
    (3) rf/gr gradients match the oracle-summed contribution of that subset when the other spins get zero upstream
        gradient -- <= 1e-4 relative for the default policy (1e-6 for 'strict');
    (4) finite-difference check of one rf sample (fp64)."""
    from mrphy import mobjs, _ops
    from oracle import bloch_oracle as orc
    N, n, nT = FULL[cfg]
    kw = {'dtype': dtype, 'device': dev}
    gen = torch.Generator().manual_seed(0)
    U = lambda *s: (torch.rand(s, generator=gen, dtype=f64) * 2 - 1)
    cube = mobjs.SpinCube((N, n, n, n), tensor([[24., 24., 24.]]), **kw)
    nM, nS = n ** 3, 128
    df, b1 = U(1, nM) * 200, U(1, nM, 2, 1) * 0.1
    b1[:, :, 0] += 1
    rf, gr = (U(N, 2, nT, 1) * 0.1).to(dtype), (U(N, 3, nT) * 2).to(dtype)
    cube.Δf_ = df.expand(N, nM)
    df, b1 = df.to(dtype), b1.to(dtype)
    sub = torch.randperm(nM, generator=gen)[:nS]
    bsel = [0] if N == 1 else [0, N // 3, N - 1]
    w = torch.zeros(N, nM, 3, dtype=f64)
    for b_ in bsel:
        w[b_, sub] = U(nS, 3)
    wd = w.to(**kw)
    b1d = b1.to(dev).expand(N, nM, 2, 1)
    c32 = lambda v: float(np.float32(v)) if dtype == f32 else v
    okw = dict(df=df[:, sub].expand(len(bsel), nS), b1=b1[:, sub].expand(len(bsel), nS, 2, 1), T1=c32(1.47), T2=c32(0.07),
               gamma=c32(4257.6), dt=c32(4e-6))
    oargs = (tensor([0., 0., 1.]).expand(len(bsel), nS, 3), rf[bsel], gr[bsel], cube.loc_.cpu()[bsel][:, sub], w[bsel][:, sub])
    ref = orc.applypulse_fwd_bwd(*oargs, **okw)
    if dtype == f64:
        runs = [(None, ATOL64, RTOL_G64)]
    else:
        ref32 = orc.applypulse_fwd_bwd(*oargs, **okw, dtype=f32)
        bound = _fp32_bound(ref32['Mo'], ref['Mo'])
        print(f'[{cfg.upper()} reference algorithm in fp32] max|dM|={mx(ref32["Mo"], ref["Mo"]):.2e} '
              f'grf rel={rel(ref32["grf"], ref["grf"]):.2e} ggr rel={rel(ref32["ggr"], ref["ggr"]):.2e}')
        # default policy: the north_star bounds.  The opt-in MUFU policies carry the unit's bias, which adds up linearly
        # over the steps (measured: mixed 4.5e-5 per 1000 steps, fast up to 7e-5): their documented bounds scale with nT
        runs = [('precise', bound, RTOL_G32), ('strict', ATOL32, 1e-6), ('mixed', bound, 6e-5 * nT / 1000),
                ('fast', 2.5 * bound, 1e-4 * nT / 1000)]
    sd = sub.to(dev)
    for pol, tolM, tolG in runs:
        _ops.set_trig_policy(pol)
        try:
            p = mobjs.Pulse(rf=rf.to(dev).requires_grad_(True), gr=gr.to(dev).requires_grad_(True), **kw)
            Mo = cube.applypulse(p, b1Map_=b1d)
            (Mo * wd).sum().backward()
        finally:
            _ops.set_trig_policy(None)
        dM, e1, e2 = mx(Mo[bsel][:, sd], ref['Mo']), rel(p.rf.grad[bsel], ref['grf']), rel(p.gr.grad[bsel], ref['ggr'])
        print(f'[{cfg.upper()} {dtype} {pol or ""}] max|dM|={dM:.2e} (bound {tolM:.2e}) grf rel={e1:.2e} ggr rel={e2:.2e}')
        assert Mo.dtype == dtype and p.rf.grad.dtype == dtype
        assert dM < tolM, (pol, dM, tolM)
        assert e1 < tolG and e2 < tolG, (pol, e1, e2)
        if N > 1:       # batch entries without upstream gradient get exactly zero waveform gradients
            rest = [i for i in range(N) if i not in bsel]
            assert float(p.rf.grad[rest].abs().max()) == 0.0 and float(p.gr.grad[rest].abs().max()) == 0.0
        del Mo
    p = mobjs.Pulse(rf=rf.to(dev), gr=gr.to(dev), **kw)
    Mn = cube.applypulse(p, b1Map_=b1d, doRelax=False).detach()
    # fp32 rounding of the state lets |M| drift by ~2e-8 per step (measured 1.3e-5 at nT=1000, 2.6e-5 at nT=2000)
    assert float((Mn.norm(dim=-1) - 1).abs().max()) < (1e-12 * nT / 1000 if dtype == f64 else 2e-5 * nT / 1000)
    del Mn
    if dtype == f64 and cfg in ('c2', 'c4'):
        p = mobjs.Pulse(rf=rf.to(dev).requires_grad_(True), gr=gr.to(dev), **kw)
        (cube.applypulse(p, b1Map_=b1d) * wd).sum().backward()
        eps, t0, b0 = 1e-6, 417, bsel[-1]
        f = lambda r: float((cube.applypulse(mobjs.Pulse(rf=r, gr=gr.to(dev), **kw), b1Map_=b1d).detach() * wd).sum())
        rp, rm = rf.to(dev).clone(), rf.to(dev).clone()
        rp[b0, 0, t0, 0] += eps
        rm[b0, 0, t0, 0] -= eps
        fd = (f(rp) - f(rm)) / (2 * eps)
        assert abs(fd - float(p.rf.grad[b0, 0, t0, 0])) < 1e-5 * max(1.0, abs(fd))


def test_rfgr2beff_kernel_and_its_chain_rule(dev):
    """CUDA rfgr2beff == the torch expressions of beffective.py:137-167, forward and every gradient
    (rf, gr, loc, Δf, b1Map, γ), with and without b1Map / coil dim, and on a 3-D Nd."""
    from mrphy import beffective
    gen = torch.Generator().manual_seed(4)
    U = lambda *s: (torch.rand(s, generator=gen, dtype=f64) * 2 - 1)
    # nT = 9 reads dL/dBeff rows straight from global memory; nT = 260 (two 256-step blocks) stages them by TMA
    for (Nd, nC, has_b1), nT in itertools.product((((7,), 2, True), ((3, 2, 2), 0, False), ((5,), 3, False), ((6,), 0, True)),
                                                  (9, 260)):
        N = 2
        rf = U(N, 2, nT, nC) if nC else U(N, 2, nT)
        ins = dict(rf=rf, gr=U(N, 3, nT), loc=U(N, *Nd, 3) * 5, df=U(N, *Nd) * 100,
                   b1=(U(N, *Nd, 2, nC) if nC else U(N, *Nd, 2)) if has_b1 else None, gam=4257.6 * (1 + 0.1 * U(N, *Nd)))
        w = U(N, *Nd, nT, 3)
        res = {}
        for where in ('cpu', 'cuda'):
            t = {k: (None if v is None else v.detach().clone().to(where).requires_grad_(True)) for k, v in ins.items()}
            fn = beffective.rfgr2beff if where == 'cuda' else torch_ref.rfgr2beff
            beff = fn(t['rf'], t['gr'], t['loc'], Δf=t['df'], b1Map=t['b1'], γ=t['gam'])
            (beff * w.to(where)).sum().backward()
            res[where] = [beff.detach().cpu()] + [None if v is None else v.grad.cpu() for v in t.values()]
        for a, b in zip(res['cpu'], res['cuda']):
            assert (a is None) == (b is None)
            if a is not None:
                assert a.shape == b.shape and rel(b, a) < 1e-12


def test_beff2ab_kernel(dev, golden):
    """CUDA beff2ab == reference A/B (tests/test_slowsims.py:60,77-84: blochsim_ab(M0, A, B) == Mo0)."""
    from mrphy import beffective, slowsims
    g = golden('kat3')
    beff = beffective.rfgr2beff(T(g['rf'], dev, f64), T(g['gr'], dev, f64), T(g['loc'], dev, f64),
                                Δf=T(g['df'], dev, f64), b1Map=T(g['b1'], dev, f64), γ=T(g['gamma'], dev, f64))
    dt, T1, T2 = T(g['dt'], dev, f64), T(g['T1'], dev, f64), T(g['T2'], dev, f64)
    A, B = beffective.beff2ab(beff, E1=torch.exp(-dt / T1), E2=torch.exp(-dt / T2), γ=T(g['gamma'], dev, f64), dt=dt)
    assert mx(A, g['A']) < 1e-12 and mx(B, g['B']) < 1e-12
    assert mx(slowsims.blochsim_ab(T(g['M0'], dev, f64), A, B), g['Mo_const']) < 1e-12
    g2 = golden('rand_mc')
    dtb = T(g2['in_dt'], dev, f64).reshape(-1, 1)
    A, B = beffective.beff2ab(T(g2['beff_f64'], dev, f64), E1=torch.exp(-dtb / T(g2['in_T1'], dev, f64)),
                              E2=torch.exp(-dtb / T(g2['in_T2'], dev, f64)), γ=T(g2['in_gam'], dev, f64),
                              dt=T(g2['in_dt'], dev, f64))
    assert mx(A, g2['A_f64']) < 1e-12 and mx(B, g2['B_f64']) < 1e-12
    A32, B32 = beffective.beff2ab(T(g2['beff_f64'], dev, f32), E1=torch.exp(-dtb / T(g2['in_T1'], dev, f64)).float(),
                                  E2=torch.exp(-dtb / T(g2['in_T2'], dev, f64)).float(), γ=T(g2['in_gam'], dev, f32),
                                  dt=T(g2['in_dt'], dev, f32))
    assert A32.dtype == f32 and mx(A32, g2['A_f64']) < 5e-5 and mx(B32, g2['B_f64']) < 5e-5


def test_gradients_through_beff2ab_equal_blochsim_goldens(dev, golden):
    """tests/test_slowsims.py:86-96: d/d(rf, gr, M0) of sum(w * blochsim_ab(M0, *beff2ab(beff))) equals the gradients
    through blochsim -- here against the reference's own gradients stored in the golden fixture."""
    from mrphy import beffective, slowsims
    g = golden('rand_mc')
    t = {k[3:]: T(v, dev, f64) for k, v in g.items() if k.startswith('in_')}
    rf, gr, M0 = (t[k].requires_grad_(True) for k in ('rf', 'gr', 'M0'))
    beff = beffective.rfgr2beff(rf, gr, t['loc'], Δf=t['df'], b1Map=t['b1'], γ=t['gam'])
    dtb = t['dt'].reshape(-1, 1)
    A, B = beffective.beff2ab(beff, E1=torch.exp(-dtb / t['T1']), E2=torch.exp(-dtb / t['T2']), γ=t['gam'], dt=t['dt'])
    Mo = slowsims.blochsim_ab(M0, A, B)
    (Mo * t['w']).sum().backward()
    assert mx(Mo, g['Mo_f64']) < 1e-12
    assert rel(rf.grad, g['grf_f64']) < 1e-10 and rel(gr.grad, g['ggr_f64']) < 1e-10
    assert rel(M0.grad, g['gM0_slow_f64']) < 1e-10


@pytest.mark.parametrize('case', ['typical', 'strong', 'E0', 'norelax'])
@pytest.mark.parametrize('dtype', [f64, f32])
def test_beff2ab_adjoint_kernel(dev, case, dtype):
    """dL/d(beff, E1, E2, γ, dt) of the CUDA beff2ab adjoint == autograd through the reference's time loop
    (beffective.py:88-103, restated in tests/torch_ref.py).  'strong' relaxation shortens the checkpoint interval,
    'E0' (the upstream default E1=E2=0) takes the division-free K=1 mode, 'norelax' is E=1."""
    from mrphy import beffective
    gen = torch.Generator().manual_seed(11)
    U = lambda *s: (torch.rand(s, generator=gen, dtype=f64) * 2 - 1)
    N, Nd, nT = 2, (3, 5), 150
    beff = U(N, *Nd, nT, 3) * torch.tensor([0.1, 0.1, 2.0], dtype=f64)
    γ = 4257.6 * (1 + 0.1 * U(N, *Nd))
    dt = 4e-6 * (1 + 0.2 * U(N))
    if case == 'typical':
        E1, E2 = torch.exp(-4e-6 / (1.0 + 0.3 * U(N, *Nd))), torch.exp(-4e-6 / (0.07 + 0.02 * U(N, *Nd)))
    elif case == 'strong':
        E1, E2 = 0.9 + 0.05 * U(N, 1, 1), 0.8 + 0.1 * U(1, *Nd)
    elif case == 'E0':
        E1, E2 = torch.tensor(0., dtype=f64), torch.tensor(0.5, dtype=f64)
    else:
        E1, E2 = torch.tensor(1., dtype=f64), torch.ones(N, 1, 1, dtype=f64)
    wA, wB = U(N, *Nd, 3, 3), U(N, *Nd, 3)
    res = {}
    for where in ('ref', 'cuda'):
        d, ty = ('cpu', f64) if where == 'ref' else (dev, dtype)
        # both sides start from the inputs as rounded to the working type (1 - E1 ~ 4e-6 has few bits left in fp32)
        t = [x.detach().clone().to(dtype).to(device=d, dtype=ty).requires_grad_(True) for x in (beff, E1, E2, γ, dt)]
        if where == 'ref':
            A, B = torch_ref.beff2ab(*t)
        else:
            A, B = beffective.beff2ab(t[0], E1=t[1], E2=t[2], γ=t[3], dt=t[4])
        ((A * wA.to(device=d, dtype=ty)).sum() + (B * wB.to(device=d, dtype=ty)).sum()).backward()
        res[where] = [A.detach().cpu().double(), B.detach().cpu().double()] + [x.grad.cpu().double() for x in t]
    tol = 1e-10 if dtype == f64 else 2e-3      # fp32: nT=150 steps of rounding in both state and adjoint
    for a, b in zip(res['ref'], res['cuda']):   # (+1e-30: with E2 = 0.5, A ~ 0.5^150 underflows in fp32)
        assert a.shape == b.shape and float((b - a).abs().max()) <= tol * float(a.abs().max()) + 1e-30


@pytest.mark.parametrize('dtype', [f64, f32])
def test_beff2uphi_kernel_and_adjoint(dev, dtype):
    """CUDA beff2uϕ == F.normalize / -norm·γ2πdt (beffective.py:35-36), values and both gradients, including a
    vanishing field, a broadcast γ2πdt and an xyz axis that is not the last one."""
    from mrphy import beffective
    gen = torch.Generator().manual_seed(12)
    U = lambda *s: (torch.rand(s, generator=gen, dtype=f64) * 2 - 1)
    for shape, gshape, dim in (((2, 4, 5, 3), (2, 1, 5), -1), ((3, 7, 3), (), -1), ((2, 3, 6), (2, 1), 1), ((1, 3), (1,), -1)):
        b = U(*shape)
        if dim == -1 and b.ndim > 2:
            b[0, 0] = 0                      # zero field: U = 0, Φ = 0, finite gradients
        g = U(*gshape) + 2
        wU, wP = U(*shape), U(*(shape[:dim % len(shape)] + shape[dim % len(shape) + 1:]))
        res = {}
        for where in ('ref', 'cuda'):
            d, ty = ('cpu', f64) if where == 'ref' else (dev, dtype)
            bt, gt = (x.detach().clone().to(device=d, dtype=ty).requires_grad_(True) for x in (b, g))
            fn = torch_ref.beff2uphi if where == 'ref' else beffective.beff2uϕ
            Uo, P = fn(bt, gt, dim=dim)
            ((Uo * wU.to(device=d, dtype=ty)).sum() + (P * wP.to(device=d, dtype=ty)).sum()).backward()
            res[where] = [x.detach().cpu().double() for x in (Uo, P, bt.grad, gt.grad)]
        for a, c in zip(res['ref'], res['cuda']):
            assert a.shape == c.shape and mx(c, a) < (1e-12 if dtype == f64 else 2e-5) * max(1.0, float(a.abs().max()))
    with torch.no_grad():                    # Φ only / U only consumers
        bt = U(2, 5, 3).to(dev).requires_grad_(True)
    Uo, P = beffective.beff2uϕ(bt, torch.tensor(2., dtype=f64, device=dev))
    P.sum().backward()
    assert mx(bt.grad, -2 * torch.nn.functional.normalize(bt.detach(), dim=-1)) < 1e-12


def test_standalone_operators_against_reference_goldens(dev, golden):
    """beff2uϕ, rfgr2beff (outputs and EVERY gradient: rf, gr, loc, Δf, b1Map, γ -- including a single-coil b1Map
    broadcast over multi-coil rf and a multi-coil b1Map with rf without a coil dim, beffective.py:153-165) and beff2ab with
    its gradients: the CUDA operators against outputs and autograd gradients of the UNMODIFIED reference
    (tests/golden/standalone.npz)."""
    from mrphy import beffective
    g = golden('standalone')
    near = lambda a, b, tol=1e-11: a.shape == tuple(np.shape(b)) and mx(a, b) <= tol * max(1.0, float(np.abs(b).max()))
    G = lambda k, grad=True: T(g[k], dev, f64).requires_grad_(grad)
    beff, gg = G('uphi_beff'), G('uphi_g')
    U, P = beffective.beff2uϕ(beff, gg)
    assert near(U, g['uphi_U']) and near(P, g['uphi_Phi'])
    ((U * G('uphi_wU', False)).sum() + (P * G('uphi_wP', False)).sum()).backward()
    assert near(beff.grad, g['uphi_gbeff']) and near(gg.grad, g['uphi_gg'])
    for tag in ('mc', 'b1bc', 'rfbc', 'nob1', 'sc'):
        t = {k: G(f'b_{tag}_{k}') for k in ('rf', 'gr', 'loc', 'df', 'gam', 'b1') if f'b_{tag}_{k}' in g}
        be = beffective.rfgr2beff(t['rf'], t['gr'], t['loc'], Δf=t['df'], b1Map=t.get('b1'), γ=t['gam'])
        assert near(be, g[f'b_{tag}_beff']), tag
        (be * G(f'b_{tag}_w', False)).sum().backward()
        for k, v in t.items():
            assert near(v.grad, g[f'b_{tag}_g{k}']), (tag, k)
    bf, E1, E2 = G('ab_beff'), G('ab_E1'), G('ab_E2')
    A, B = beffective.beff2ab(bf, E1=E1, E2=E2, γ=tensor(4257.6, dtype=f64), dt=tensor(4e-6, dtype=f64))
    assert near(A, g['ab_A']) and near(B, g['ab_B'])
    ((A * G('ab_wA', False)).sum() + (B * G('ab_wB', False)).sum()).backward()
    assert near(bf.grad, g['ab_gbeff'], 1e-9) and near(E1.grad, g['ab_gE1'], 1e-9) and near(E2.grad, g['ab_gE2'], 1e-9)


def test_applypulse_with_broadcast_b1map_on_both_paths(dev, golden):
    """A single-coil b1Map with multi-coil rf, and a multi-coil b1Map with rf without a coil dim, through the fused path
    and (loc requiring grad) through the explicit-field path: both equal the reference chain's field + the oracle."""
    from mrphy import mobjs
    from oracle import bloch_oracle as orc
    g = golden('standalone')
    kw = {'dtype': f64, 'device': dev}
    for tag in ('b1bc', 'rfbc'):
        rf, gr, loc, b1 = (T(g[f'b_{tag}_{k}'], dev, f64) for k in ('rf', 'gr', 'loc', 'b1'))
        N, nM = loc.shape[0], loc.shape[1]
        # the oracle takes matching coil dims: spell the broadcast out (expanded b1Map / coil-summed b1Map)
        rf_o = g[f'b_{tag}_rf'] if tag == 'b1bc' else g[f'b_{tag}_rf'][..., None]
        b1_o = np.broadcast_to(g[f'b_{tag}_b1'], (N, nM, 2, 3)) if tag == 'b1bc' else g[f'b_{tag}_b1'].sum(-1, keepdims=True)
        Mo_ref = orc.blochsim_fwd(tensor([0., 0., 1.]).expand(N, nM, 3),
                                  orc.rfgr2beff(rf_o, g[f'b_{tag}_gr'], g[f'b_{tag}_loc'], b1=b1_o), 1.47, 0.07)
        sp = mobjs.SpinArray((N, nM), **kw)
        p = mobjs.Pulse(rf=rf, gr=gr, **kw)
        M1 = sp.applypulse(p, loc_=loc, b1Map_=b1)
        M2 = sp.applypulse(p, loc_=loc.clone().requires_grad_(True), b1Map_=b1)        # routes through rfgr2beff + blochsim
        assert mx(M1, Mo_ref) < 1e-12 and mx(M2, Mo_ref) < 1e-12


@pytest.mark.parametrize('dtype', [f64, f32])
def test_rfclamp_sclamp_kernels_match_reference(dev, golden, dtype):
    """utils.rfclamp / utils.sclamp on CUDA tensors (one launch each way, csrc/design_ops.cu: clamp_waveform_kernel)
    against the unmodified reference's outputs and autograd gradients (tests/golden/standalone.npz)."""
    from mrphy import utils, _cabi
    g = golden('standalone')
    tol = 1e-12 if dtype == f64 else 2e-6
    near = lambda a, b: mx(a, b) <= tol * max(1.0, float(np.abs(b).max()))
    for tag in ('sc', 'mc'):
        rf = T(g[f'cl_{tag}_rf'], dev, dtype).requires_grad_(True)
        n0 = _cabi.launch_counter
        out = utils.rfclamp(rf, T(g[f'cl_{tag}_rfmax'], dev, dtype))
        (out * T(g[f'cl_{tag}_w'], dev, dtype)).sum().backward()
        assert _cabi.launch_counter - n0 == 2                       # one launch forward, one backward
        assert out.dtype == dtype and near(out, g[f'cl_{tag}_out']) and near(rf.grad, g[f'cl_{tag}_grf'])
        assert (np.abs(g[f'cl_{tag}_out'] - g[f'cl_{tag}_rf']) > 0).any()   # the fixture does clamp something
    s = T(g['cl_s'], dev, dtype).requires_grad_(True)
    out = utils.sclamp(s, T(g['cl_smax'], dev, dtype))
    (out * T(g['cl_ws'], dev, dtype)).sum().backward()
    assert near(out, g['cl_sout']) and near(s.grad, g['cl_gs'])
    # scalar limits and the CPU expressions agree with the kernels
    rf = T(g['cl_sc_rf'], dev, dtype)
    lim = tensor(0.15, dtype=dtype)
    assert mx(utils.rfclamp(rf, lim), utils.rfclamp(rf.cpu(), lim)) <= tol
    assert mx(utils.sclamp(s.detach(), tensor(9e3)), utils.sclamp(s.detach().cpu(), tensor(9e3))) == 0.0


@pytest.mark.parametrize('dtype', [f64, f32])
def test_applysequence_matches_chained_reference(dev, golden, dtype):
    """pulse -> freeprec -> pulse on a masked SpinCube (SURVEY 8f-1): `applysequence` against the unmodified reference
    chained through doUpdate (forward, tests/golden/sequence.npz) and its autograd gradients w.r.t. both pulses; the same
    values from chaining our own applypulse / freeprec; no host synchronisation; and the whole sequence + loss + backward
    replayed from ONE CUDA graph reproduces the eager gradients bit for bit."""
    from mrphy import mobjs, graphs
    g = golden('sequence')
    kw = {'dtype': dtype, 'device': dev}
    tolM, tolG = (1e-12, 1e-9) if dtype == f64 else (1e-5, 1e-4)

    def build():
        cube = mobjs.SpinCube((2, 4, 3, 3), T(g['fov'], dev, dtype), mask=tensor(g['mask'], device=dev), ofst=T(g['ofst'], dev, dtype),
                              Δf_=T(g['df'], dev, dtype), T1_=T(g['T1'], dev, dtype), T2_=T(g['T2'], dev, dtype), **kw)
        p1 = mobjs.Pulse(rf=T(g['rf1'], dev, dtype).requires_grad_(True), gr=T(g['gr1'], dev, dtype).requires_grad_(True),
                         dt=tensor(4e-6, dtype=f64), **kw)
        p2 = mobjs.Pulse(rf=T(g['rf2'], dev, dtype).requires_grad_(True), gr=T(g['gr2'], dev, dtype).requires_grad_(True),
                         dt=tensor(8e-6, dtype=f64), **kw)
        return cube, p1, p2

    cube, p1, p2 = build()
    b1, dur, w = T(g['b1'], dev, dtype), T(g['dur'], dev, dtype), T(g['w'], dev, dtype)
    cube.applysequence([p1, dur, p2], b1Map_=b1)      # first use reads min(T1, T2) once (cached per tensor afterwards)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')           # from here on: no device->host read at all
    try:
        Mc = cube.applysequence([p1, dur, p2], b1Map_=b1)
        (Mc * w).sum().backward()
    finally:
        torch.cuda.set_sync_debug_mode('default')
    assert mx(Mc, g['Mc']) < tolM
    for got, key in ((p1.rf.grad, 'grf1'), (p1.gr.grad, 'ggr1'), (p2.rf.grad, 'grf2'), (p2.gr.grad, 'ggr2')):
        assert rel(got, g[key]) < tolG, key
    # chaining the object methods gives the same intermediate and final states
    c2, q1, q2 = build()
    c2.applypulse(q1, b1Map_=b1, doUpdate=True)
    assert mx(c2.M_, g['Ma']) < tolM
    c2.freeprec(dur, doUpdate=True)
    assert mx(c2.M_, g['Mb']) < tolM
    assert mx(c2.applypulse(q2, b1Map_=b1), Mc) == 0.0
    # one CUDA graph for the whole sequence + loss + backward
    eager = [x.grad.clone() for x in (p1.rf, p1.gr, p2.rf, p2.gr)]
    del Mc
    step = graphs.capture(lambda: (cube.applysequence([p1, dur, p2], b1Map_=b1) * w).sum().backward(),
                          params=(p1.rf, p1.gr, p2.rf, p2.gr))
    step.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b.grad) for a, b in zip(eager, (p1.rf, p1.gr, p2.rf, p2.gr)))


def test_integration_md_stub_runs(dev):
    """The ctypes stub INTEGRATION.md section 2 shows a maintainer (struct mirrors + `BlochSim.forward` over
    `mrphy_blochsim_beff_fwd`) is executed verbatim -- only the library path is filled in -- and reproduces the oracle."""
    import re
    from mrphy import _cabi
    from oracle import bloch_oracle as orc
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    md = open(os.path.join(root, 'INTEGRATION.md')).read()
    sec = md[md.index('## 2.'):md.index('## 3.')]
    code = re.search(r'```python\n(.*?)```', sec, flags=re.S).group(1)
    assert "'.../libmrphy_b200.so'" in code
    ns = {}
    exec(code.replace("'.../libmrphy_b200.so'", repr(_cabi.LIB_PATH)), ns)
    p = _random_problem(13, 2, 70, 45, 1, has_b1=True, relax=True)
    beff = orc.rfgr2beff(p['rf'], p['gr'], p['loc'], df=p['df'], b1=p['b1'], gamma=p['gam'])
    col = lambda x: x.to(dev).reshape(x.shape[0], -1)                      # (N|1, nM|1) as the stub's _param expects
    Mo = ns['BlochSim'].apply(p['M0'].to(dev), beff.to(dev), col(p['T1']), col(p['T2']), col(p['gam']),
                              p['dt'].to(dev).reshape(1, 1))
    assert mx(Mo, orc.blochsim_fwd(p['M0'], beff, p['T1'], p['T2'], p['gam'], p['dt'])) < ATOL64


def test_interpT_on_device_goldens_no_sync_and_gradient(dev, golden):
    """Pulse.interpT (linear) on CUDA tensors: the reference's values (tests/test_mobjs.py:160-195 and fixtures from the
    unmodified reference, incl. the float-// length quirk and the fp32 1999-vs-2000 case), NO device->host read, and
    with differentiable=True the gradient of the resampling (against the oracle's numpy interpolation as a matrix)."""
    from mrphy import mobjs, dt0
    from oracle import bloch_oracle as orc
    g = golden('interp')
    kw = {'dtype': f64, 'device': dev}
    p = mobjs.Pulse(rf=T(g['a_rf'], dev, f64), gr=T(g['a_gr'], dev, f64), dt=dt0, **kw)
    p2 = mobjs.Pulse(rf=T(g['b_rf'], dev, f64), gr=T(g['b_gr'], dev, f64), dt=dt0, **kw)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')       # no device->host read and no synchronous host->device copy from here on
    try:
        q = p.interpT(dt=dt0 * 5)
        q2 = p2.interpT(dt=tensor(2e-6, dtype=f64))
        q2b = q2.interpT(dt=tensor(1e-6, dtype=f64))          # resampling a resampled pulse: its dt is host-known too
    finally:
        torch.cuda.set_sync_debug_mode('default')
    assert q.rf.is_cuda and q.rf.cpu().numpy() == pytest.approx(np.array([[[0.04, 0.09], [0.06, 0.01]]]), abs=1e-9)
    assert q.gr.cpu().numpy() == pytest.approx(np.array([[[0.04, 0.09], [0.06, 0.01], [0.1, 0.1]]]), abs=1e-9)
    assert q2.rf.shape[2] == 19 and mx(q2.rf, g['b_rf_new']) < 1e-12 and mx(q2.gr, g['b_gr_new']) < 1e-12
    assert q2b.rf.shape[2] == int((19 * 2e-6) // 1e-6) and mx(q2b.rf, orc.interp_linear(g['b_rf_new'], 2e-6, 1e-6)) < 1e-12
    p3f = mobjs.Pulse(rf=T(g['c_rf'], dev, f32), gr=T(g['c_gr'], dev, f32), dt=tensor(20e-6, dtype=f64), dtype=f32, device=dev)
    q3f = p3f.interpT(dt=tensor(4e-6, dtype=f64))
    assert q3f.rf.shape[2] == 199 and mx(q3f.rf, g['c32_rf_new']) < 1e-6 and mx(q3f.gr, g['c32_gr_new']) < 1e-6
    # gradient: q = J x with J the (linear) interpolation matrix, so dL/dx = J^T w
    rf = T(g['b_rf'], dev, f64).requires_grad_(True)
    gr = T(g['b_gr'], dev, f64).requires_grad_(True)
    pd = mobjs.Pulse(rf=rf, gr=gr, dt=dt0, **kw)
    qd = pd.interpT(dt=tensor(2e-6, dtype=f64), differentiable=True)
    assert not pd.interpT(dt=tensor(2e-6, dtype=f64)).rf.requires_grad and qd.rf.requires_grad
    gen = torch.Generator().manual_seed(1)
    w = torch.rand(qd.rf.shape, generator=gen, dtype=f64)
    (qd.rf * w.to(dev)).sum().backward()
    nT = rf.shape[2]
    J = orc.interp_linear(np.eye(nT)[None], 4e-6, 2e-6)[0]                 # (nT, nT_new): column j = weights of sample j
    want = np.einsum('tj,ncj->nct', J, w.numpy())
    assert mx(rf.grad, want) < 1e-12 and gr.grad is None


def test_multiscale_design_loop_through_public_api(dev):
    """The use the reference is built for (BASELINE config C3 in miniature): optimise a pulse through its
    re-parametrisation (utils.tρθ2rf / ts2s / s2g), refine it with Pulse.interpT on the device, keep optimising.
    The loss must fall at both scales, and the interpolated pulse must reproduce the coarse pulse's magnetisation
    to first order (same waveform, 5x finer steps)."""
    from mrphy import mobjs, utils
    kw = {'dtype': f32, 'device': dev}
    cube = mobjs.SpinCube((1, 8, 8, 8), tensor([[24., 24., 24.]]), **kw)
    cube.Δf = (torch.rand(1, 8, 8, 8, generator=torch.Generator().manual_seed(0)) * 100 - 50).to(dev)
    tgt = tensor([0., 1., 0.], **kw)

    def loss_of(pulse):
        cube.M = tensor([0., 0., 1.], **kw)
        return ((cube.applypulse(pulse, doEmbed=False) - tgt) ** 2).mean()

    def descend(p0, iters, lr):
        rfmax, smax = p0.rfmax, p0.smax
        tρ, θ = (x.detach().clone().requires_grad_(True) for x in utils.rf2tρθ(p0.rf, rfmax))
        ts = utils.s2ts(utils.g2s(p0.gr, p0.dt), smax).detach().clone().requires_grad_(True)
        hist = []
        for _ in range(iters):
            p = mobjs.Pulse(rf=utils.tρθ2rf(tρ, θ, rfmax), gr=utils.s2g(utils.ts2s(ts, smax), p0.dt), dt=p0.dt, **kw)
            L = loss_of(p)
            L.backward()
            hist.append(float(L.detach()))
            with torch.no_grad():
                for v in (tρ, θ, ts):
                    v -= lr * v.grad / (v.grad.abs().max() + 1e-12)
                    v.grad = None
        return p, hist

    gen = torch.Generator().manual_seed(1)
    nT = 40
    rf0 = (torch.rand(1, 2, nT, generator=gen) * 2 - 1) * 0.02
    gr0 = torch.cumsum((torch.rand(1, 3, nT, generator=gen) * 2 - 1) * 0.02, dim=2)
    coarse = mobjs.Pulse(rf=rf0, gr=gr0, dt=tensor(20e-6, dtype=f64), **kw)
    coarse, h1 = descend(coarse, 6, 0.05)
    assert h1[-1] < h1[0]
    fine = mobjs.Pulse(rf=coarse.rf.detach().double(), gr=coarse.gr.detach().double(), dt=tensor(20e-6, dtype=f64),
                       dtype=f64, device=dev).interpT(dt=tensor(4e-6, dtype=f64)).to(device=dev, dtype=f32)
    assert fine.rf.shape[2] == 5 * nT and fine.rf.device.type == 'cuda'
    with torch.no_grad():
        assert abs(float(loss_of(fine)) - float(loss_of(coarse))) < 0.05
    _, h2 = descend(fine, 4, 0.02)
    assert h2[-1] < h2[0]


def _design_problem(dev, dtype, nC, seed=3, N=2, nM=301, nT=333):
    """Design variables (tρ, θ, ts), limits, and a spin set; sizes ragged on purpose (nT not a multiple of 32)."""
    gen = torch.Generator().manual_seed(seed)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    shp = (N, 1, nT, nC) if nC > 1 else (N, 1, nT)
    d = dict(rho=U(*shp) * 2, theta=U(*shp) * 3, ts=U(N, 3, nT) * 1.5,
             rfmax=(0.15 + 0.05 * U(N, nC).abs()) if nC > 1 else (0.15 + 0.05 * U(N).abs()),
             smax=1.2e4 + 2e3 * U(N, 3).abs(), dt=tensor([4e-6], dtype=f64))
    p = _random_problem(seed + 40, N, nM, nT, nC if nC > 1 else 1, has_b1=True, relax=True)
    return {k: v.to(dtype).to(f64) for k, v in d.items()}, p


def _design_step(dev, dtype, d, p, mode, fuse, extra_penalty=False, retain=False, hook=None):
    """loss = Σ w·Mo(applypulse(chain(tρ, θ, ts))) -> (Mo, dL/dtρ, dL/dθ, dL/dts, backward launches)."""
    from mrphy import utils, _ops, _cabi
    os.environ['MRPHY_B200_FUSE_DESIGN'] = '1' if fuse else '0'
    try:
        t = {k: T(v.numpy(), dev, dtype) for k, v in d.items()}
        rho, theta, ts = (t[k].clone().requires_grad_(True) for k in ('rho', 'theta', 'ts'))
        if mode == 'joint':
            rf, gr = utils.tρθts2rfgr(rho, theta, ts, t['rfmax'], t['smax'], t['dt'])
        elif mode == 'split':                    # two chains, logit amplitude, slew given directly
            rf, gr = utils.lρθ2rf(rho, theta, t['rfmax']), utils.s2g(ts, t['dt'])
        elif mode == 'rf_only':                  # gr is a plain leaf
            rf, gr = utils.tρθ2rf(rho, theta, t['rfmax']), ts
        else:                                    # 'gr_only': rf is a plain leaf
            rf = torch.cat([rho, theta], dim=1).mul(0.05).detach().requires_grad_(True)
            gr = utils.ts2g(ts, t['smax'], t['dt'])
        if retain:
            rf.retain_grad()
        if hook is not None:
            rf.register_hook(hook)
        q = {k: (None if v is None else T(v.numpy(), dev, dtype)) for k, v in p.items()}
        Mo = _ops.fused_applypulse(q['M0'], rf, gr, q['loc'], Δf_=q['df'], b1Map_=q['b1'], T1_=q['T1'], T2_=q['T2'],
                                   γ_=T(p['gam'].numpy(), dev, f64), dt=T(p['dt'].numpy(), dev, f64))
        loss = (Mo * q['w']).sum()
        if extra_penalty:                        # a second consumer of rf: its gradient must add up at the leaves
            loss = loss + 3.0 * (rf ** 2).sum()
        n0 = _cabi.launch_counter
        loss.backward()
        launches = _cabi.launch_counter - n0
        grads = (rho.grad, theta.grad, ts.grad)
        leaf_rf = rf.grad if (retain or mode == 'gr_only') else None
        return Mo.detach(), grads, launches, leaf_rf
    finally:
        os.environ.pop('MRPHY_B200_FUSE_DESIGN', None)


@pytest.mark.parametrize('dtype', [f64, f32])
@pytest.mark.parametrize('mode,nC', [('joint', 1), ('joint', 2), ('split', 1), ('split', 4), ('rf_only', 1), ('gr_only', 1)])
def test_design_adjoint_fused_into_gradient_epilogue(dev, dtype, mode, nC):
    """SURVEY 8f-2: waveforms that come out of utils.tρθ2rf / lρθ2rf / s2g / ts2g / tρθts2rfgr carry their design variables,
    and `applypulse`'s backward evaluates dL/dtρ, dL/dθ, dL/dts in the tail of its own gradient epilogue
    (grad_finalize_design_kernel) -- one launch fewer, same numbers.  Checked against (a) the two-stage path (simulation
    backward, then the chain's own adjoint kernel, itself pinned to the reference's autograd in
    test_design_waveform_kernel_matches_reference) and (b) the fp64 oracle's dL/drf, dL/dgr pushed through the reference
    chain's torch expressions on the CPU.  Tolerance: fp64 1e-9 relative, fp32 1e-4 relative (north_star's gradient bound);
    fused vs two-stage 1e-12 / 1e-6 relative (the same double arithmetic on the same waveform gradients)."""
    from oracle import bloch_oracle as orc
    from mrphy import utils
    d, p = _design_problem(dev, dtype, nC)
    Mo_f, g_f, n_f, _ = _design_step(dev, dtype, d, p, mode, fuse=True)
    Mo_u, g_u, n_u, _ = _design_step(dev, dtype, d, p, mode, fuse=False)
    assert torch.equal(Mo_f, Mo_u)
    assert n_f == n_u - (2 if mode == 'split' else 1), (n_f, n_u)       # the chain's backward launch(es) are gone
    tol_same = 1e-12 if dtype == f64 else 1e-6
    for a, b in zip(g_f, g_u):
        assert (a is None) == (b is None)
        if a is not None:
            assert rel(a, b) < tol_same, (mode, rel(a, b))
    # (b) oracle: chain on the CPU in fp64 torch expressions (the reference formulas), simulation gradients from the oracle
    rho, theta, ts = (d[k].clone().requires_grad_(True) for k in ('rho', 'theta', 'ts'))
    if mode == 'joint':
        rf, gr = utils.tρθ2rf(rho, theta, d['rfmax']), utils.s2g(utils.ts2s(ts, d['smax']), d['dt'])
    elif mode == 'split':
        rf, gr = utils.lρθ2rf(rho, theta, d['rfmax']), utils.s2g(ts, d['dt'])
    elif mode == 'rf_only':
        rf, gr = utils.tρθ2rf(rho, theta, d['rfmax']), ts
    else:
        rf, gr = torch.cat([rho, theta], dim=1).mul(0.05), utils.ts2g(ts, d['smax'], d['dt'])
    rf32, gr32 = rf.detach().to(dtype).to(f64), gr.detach().to(dtype).to(f64)     # what the kernels were handed
    ref = orc.applypulse_fwd_bwd(p['M0'], rf32, gr32, p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'], T2=p['T2'],
                                 gamma=p['gam'], dt=p['dt'])
    torch.autograd.backward([rf, gr], [torch.as_tensor(ref['grf']).reshape(rf.shape), torch.as_tensor(ref['ggr'])])
    tol = RTOL_G64 if dtype == f64 else RTOL_G32
    want = (rho.grad, theta.grad, ts.grad)
    if mode == 'gr_only':
        want = (None, None, ts.grad)
        g_f = (None, None, g_f[2])
    for name, a, b in zip(('rho', 'theta', 'ts'), g_f, want):
        if b is not None:
            print(f'[design tail {mode} nC={nC} {dtype}] d{name}: rel {rel(a, b):.2e}')
            assert rel(a, b) < tol, (name, rel(a, b))


def test_design_tail_second_consumer_retain_grad_and_graph_replay(dev):
    """(1) rf also feeds a penalty term: the simulation's share arrives through the fused tail, the penalty's through the
    chain's own backward, and autograd adds them at the leaves.  (2) `rf.retain_grad()` or a hook on rf: the caller wants dL/drf
    itself, so the two-stage path runs and rf.grad is filled / the hook fires.  (3) a captured step replays with the finished-CTA counters reset by the
    kernels themselves: three replays, bit-identical gradients."""
    from mrphy import utils, _ops, graphs
    d, p = _design_problem(dev, f32, 1, seed=9, N=1, nM=700, nT=130)
    _, g_f, _, _ = _design_step(dev, f32, d, p, 'joint', fuse=True, extra_penalty=True)
    _, g_u, _, _ = _design_step(dev, f32, d, p, 'joint', fuse=False, extra_penalty=True)
    for a, b in zip(g_f, g_u):
        assert rel(a, b) < 1e-6
    _, g_r, n_r, rf_grad = _design_step(dev, f32, d, p, 'joint', fuse=True, retain=True)
    _, g_0, n_0, _ = _design_step(dev, f32, d, p, 'joint', fuse=False)
    assert rf_grad is not None and n_r == n_0 and all(torch.equal(a, b) for a, b in zip(g_r, g_0))
    seen = []
    _, g_h, n_h, _ = _design_step(dev, f32, d, p, 'joint', fuse=True, hook=lambda g: seen.append(g.clone()))
    assert len(seen) == 1 and torch.equal(seen[0], rf_grad) and n_h == n_0      # a hook on rf still sees dL/drf
    t = {k: T(v.numpy(), dev, f32) for k, v in d.items()}
    rho, theta, ts = (t[k].clone().requires_grad_(True) for k in ('rho', 'theta', 'ts'))
    q = {k: (None if v is None else T(v.numpy(), dev, f32)) for k, v in p.items()}
    gam, dts = T(p['gam'].numpy(), dev, f64), T(p['dt'].numpy(), dev, f64)

    def step():
        rf, gr = utils.tρθts2rfgr(rho, theta, ts, t['rfmax'], t['smax'], t['dt'])
        Mo = _ops.fused_applypulse(q['M0'], rf, gr, q['loc'], Δf_=q['df'], b1Map_=q['b1'], T1_=q['T1'], T2_=q['T2'], γ_=gam,
                                   dt=dts)
        (Mo * q['w']).sum().backward()

    step()
    want = [x.grad.clone() for x in (rho, theta, ts)]
    captured = graphs.capture(step, params=(rho, theta, ts))
    for _ in range(3):
        captured.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(x.grad, w) for x, w in zip((rho, theta, ts), want))


def test_step_is_cuda_graph_capturable(dev):
    """A whole design step (applypulse forward, loss, adjoint backward) records into a CUDA graph after warm-up: no
    host synchronisation, no allocation outside torch's allocator, every launch on the capturing stream.  Replays with
    new waveform values reproduce the eager gradients bit for bit."""
    from mrphy import mobjs
    kw = {'dtype': f32, 'device': dev}
    gen = torch.Generator().manual_seed(5)
    cube = mobjs.SpinCube((1, 12, 12, 12), tensor([[24., 24., 24.]]), **kw)
    cube.Δf = (torch.rand(1, 12, 12, 12, generator=gen) * 200 - 100).to(dev)
    nT = 96
    rfs = [(torch.rand(1, 2, nT, generator=gen) * 0.2 - 0.1).to(dev) for _ in range(3)]
    grs = [(torch.rand(1, 3, nT, generator=gen) * 4 - 2).to(dev) for _ in range(3)]
    pulse = mobjs.Pulse(rf=rfs[0].clone().requires_grad_(True), gr=grs[0].clone().requires_grad_(True), **kw)
    sp, loc, df = cube.spinarray, cube.loc_, cube.Δf_
    M0 = sp.M_.clone()
    tgt = tensor([0., 1., 0.], **kw)

    def step():
        M = sp.applypulse(pulse, loc_=loc, Δf_=df)
        loss = ((M - tgt) ** 2).sum()
        loss.backward()
        return loss

    def eager(rf, gr):
        with torch.no_grad():
            pulse.rf.copy_(rf); pulse.gr.copy_(gr)
        pulse.rf.grad = pulse.gr.grad = None
        L = step()
        return L.detach().clone(), pulse.rf.grad.clone(), pulse.gr.grad.clone()

    want = [eager(rf, gr) for rf, gr in zip(rfs, grs)]
    from mrphy import graphs
    captured = graphs.capture(step, params=(pulse.rf, pulse.gr))
    for (L, grf, ggr), rf, gr in zip(want, rfs, grs):
        with torch.no_grad():
            pulse.rf.copy_(rf); pulse.gr.copy_(gr)
        static_loss = captured.replay()
        torch.cuda.synchronize()
        assert torch.equal(static_loss, L) and torch.equal(pulse.rf.grad, grf) and torch.equal(pulse.gr.grad, ggr)
    assert torch.equal(sp.M_, M0)          # doUpdate=False: the stored state is untouched


def test_host_constants_are_cached_per_object_and_version(dev):
    """`_ops.on_device`: a small CPU constant maps to ONE device tensor per (object, in-place version) -- the default
    γH / dt0 therefore cost no copy and no synchronisation per call -- and an in-place edit or a tensor that requires
    grad is never served from the cache."""
    from mrphy import _ops, dt0
    a, b = _ops.on_device(dt0, dev), _ops.on_device(dt0, dev)
    assert a is b and a.device == dev and float(a) == float(dt0)
    c = torch.tensor([1.5, 2.5], dtype=f64)
    c1 = _ops.on_device(c, dev)
    c.mul_(2)
    c2 = _ops.on_device(c, dev)
    assert c2 is not c1 and c2.tolist() == [3.0, 5.0] and c1.tolist() == [1.5, 2.5]
    g = torch.tensor(2.0, requires_grad=True)
    assert _ops.on_device(g, dev) is not _ops.on_device(g, dev) and _ops.on_device(g, dev).requires_grad
    big = torch.zeros(64)
    assert _ops.on_device(big, dev) is not _ops.on_device(big, dev)
    assert _ops.on_device(a, dev) is a and _ops.on_device(None, dev) is None


def test_freeprec_kernel(dev, golden):
    """tests/test_slowsims.py:100-122, tests/test_sims.py:145-198, tests/test_mobjs.py:133-158 on CUDA."""
    from mrphy import sims, mobjs, γH
    g = golden('freeprec')
    Mo = sims.freeprec(T(g['a_Mi'], dev, f64), T(g['a_dur'], dev, f64), T1=T(g['a_T1'], dev, f64),
                       T2=T(g['a_T2'], dev, f64), Δf=T(g['a_df'], dev, f64))
    assert mx(Mo, [[[0., -0.5, 0.5], [-0.5, 0, 0.5], [0., 0., 1.]]]) < 1e-12
    for dtype, tol in ((f64, 1e-13), (f32, 2e-6)):
        Mi = T(g['b_Mi'], dev, dtype).requires_grad_(True)
        Mo = sims.freeprec(Mi, T(g['b_dur'], dev, dtype), T1=T(g['b_T1'], dev, dtype), T2=T(g['b_T2'], dev, dtype),
                           Δf=T(g['b_df'], dev, dtype))
        (Mo * T(g['b_w'], dev, dtype)).sum().backward()
        assert Mo.dtype == dtype and mx(Mo, g['b_Mo']) < tol and mx(Mi.grad, g['b_gMi']) < tol
    Mo = sims.freeprec(T(g['b_Mi'], dev, f64), T(g['b_dur'], dev, f64))          # no relaxation, no precession
    assert mx(Mo, g['b_Mi']) == 0.0
    cube = mobjs.SpinCube((1, 3, 3, 3), tensor([[3., 3., 3.]]), T1_=tensor([[0.5 / np.log(2)]], dtype=f64),
                          T2_=tensor([[0.5 / np.log(2)]], dtype=f64), γ=γH, dtype=f64, device=dev)
    cube.M_ = tensor([0., 1., 0.])
    cube.Δf = tensor([[[1 / 4 / 0.5], [-1 / 4 / 0.5], [1]]], dtype=f64).repeat(1, 3, 1, 3)
    M = cube.freeprec(tensor(0.5, dtype=f64), doEmbed=True)
    assert M[0, 1, :, 1, :].cpu().numpy() == pytest.approx(np.array([[0.5, 0., 0.5], [-0.5, 0., 0.5], [0., -0.5, 0.5]]), abs=1e-9)


def test_spincube_api_batch_mask_multicoil(dev):
    """The object API end to end on CUDA: N=2 batch, masked cube, 3 coils with a NON-compact b1Map (N,*Nd,xy,nCoils),
    per-batch dt, doEmbed; against the oracle on the compact spins."""
    from mrphy import mobjs
    from oracle import bloch_oracle as orc
    gen = torch.Generator().manual_seed(12)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    N, Nd, nT, nC = 2, (5, 4, 3), 77, 3
    mask = torch.rand((1,) + Nd, generator=gen) > 0.3
    kw = {'dtype': f64, 'device': dev}
    cube = mobjs.SpinCube((N,) + Nd, tensor([[10., 8., 6.], [12., 8., 6.]]), mask=mask, ofst=tensor([[0., 1., 0.]]),
                          T1=1 + 0.3 * U(N, *Nd).abs(), T2=0.05 + 0.02 * U(N, *Nd).abs(), **kw)
    cube.Δf = U(N, *Nd) * 150
    b1 = U(N, *Nd, 2, nC) * 0.5
    rf, gr = (U(N, 2, nT, nC) * 0.2).to(dev).requires_grad_(True), (U(N, 3, nT) * 3).to(dev).requires_grad_(True)
    p = mobjs.Pulse(rf=rf, gr=gr, dt=tensor([4e-6, 8e-6]), **kw)
    M = cube.applypulse(p, b1Map=b1.to(dev), doEmbed=True)
    assert M.shape == (N,) + Nd + (3,) and bool(torch.isnan(M[:, ~mask[0].to(dev)]).all())
    M_ = cube.extract(M)
    w = U(N, cube.nM, 3)
    (M_ * w.to(dev)).sum().backward()
    c = lambda x: x.detach().cpu()
    ref = orc.applypulse_fwd_bwd(c(cube.M_), c(rf), c(gr), c(cube.loc_), w, df=c(cube.Δf_), b1=c(cube.extract(b1.to(dev))),
                                 T1=c(cube.T1_), T2=c(cube.T2_), gamma=c(cube.γ_), dt=c(p.dt))
    assert mx(M_, ref['Mo']) < ATOL64 and rel(rf.grad, ref['grf']) < RTOL_G64 and rel(gr.grad, ref['ggr']) < RTOL_G64
    # moving objects between devices keeps the data (Pulse.to / SpinCube.to, untested upstream)
    cpu_cube = cube.to(device=torch.device('cpu'), dtype=f64)
    assert torch.equal(cpu_cube.loc_, c(cube.loc_)) and torch.equal(cpu_cube.T1_, c(cube.T1_)) and cpu_cube.nM == cube.nM
    back = cpu_cube.to(device=dev, dtype=torch.float32)
    assert back.dtype == torch.float32 and back.is_cuda and mx(back.Δf_, cube.Δf_) < 1e-4
    assert mx(back.applypulse(p.to(device=dev, dtype=torch.float32), b1Map=b1.to(dev)), ref['Mo']) < 1e-4


def test_sixteen_coils_and_too_many(dev):
    from mrphy import _ops
    from oracle import bloch_oracle as orc
    p = _random_problem(31, 1, 40, 30, 11, has_b1=True, relax=True)
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'],
                                 T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    g = {('in_' + k): v.numpy() for k, v in p.items() if v is not None}
    Mo, gM0, grf, ggr = run_fused(g, dev, f64, p['w'].numpy())
    assert mx(Mo, ref['Mo']) < ATOL64 and rel(grf, ref['grf']) < RTOL_G64 and rel(ggr, ref['ggr']) < RTOL_G64
    q = _random_problem(32, 1, 8, 5, 17, has_b1=True, relax=False)
    with pytest.raises(RuntimeError, match='16 transmit coils'):
        run_fused({('in_' + k): v.numpy() for k, v in q.items() if v is not None}, dev, f64, q['w'].numpy())


def test_strong_relaxation_shrinks_checkpoint_interval(dev):
    """dt/T2 = 0.2: inverting the relaxation over 64 steps would amplify errors by e^12.8; the host policy picks
    K = 2 and gradients stay exact."""
    from mrphy import _ops
    from oracle import bloch_oracle as orc
    p = _random_problem(41, 1, 100, 90, 1, has_b1=True, relax=True)
    p['dt'] = tensor([1e-3], dtype=f64)
    p['T1'], p['T2'] = p['T1'] * 0 + 8e-3, p['T2'] * 0 + 5e-3
    p['rf'], p['gr'] = p['rf'] * 0.01, p['gr'] * 0.01
    assert _ops.pick_ckpt_interval(p['dt'].to(dev), p['T1'].to(dev), p['T2'].to(dev)) == 2
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'],
                                 T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    g = {('in_' + k): v.numpy() for k, v in p.items() if v is not None}
    Mo, gM0, grf, ggr = run_fused(g, dev, f64, p['w'].numpy())
    assert mx(Mo, ref['Mo']) < ATOL64 and rel(grf, ref['grf']) < 1e-8 and rel(ggr, ref['ggr']) < 1e-8
    assert rel(gM0, ref['gM0']) < 1e-8


def test_geometry_gradients_route_through_explicit_field(dev):
    """loc / Δf / b1Map that require grad: applypulse materialises Beff (CUDA rfgr2beff) and uses the explicit-Beff
    kernels, so the reference's autograd behaviour is kept; checked by finite differences."""
    from mrphy import mobjs
    gen = torch.Generator().manual_seed(8)
    U = lambda *s: torch.rand(s, generator=gen, dtype=f64) * 2 - 1
    kw = {'dtype': f64, 'device': dev}
    sp = mobjs.SpinArray((1, 6), **kw)
    p = mobjs.Pulse(rf=(U(1, 2, 20) * 0.2).to(dev), gr=(U(1, 3, 20) * 3).to(dev), **kw)
    loc, df = (U(1, 6, 3) * 5).to(dev).requires_grad_(True), (U(1, 6) * 100).to(dev).requires_grad_(True)
    w = U(1, 6, 3).to(dev)
    f = lambda l, d: (sp.applypulse(p, loc_=l, Δf_=d) * w).sum()
    f(loc, df).backward()
    eps = 1e-6
    for t, idx in ((loc, (0, 2, 1)), (df, (0, 4))):
        tp, tm = t.detach().clone(), t.detach().clone()
        tp[idx] += eps
        tm[idx] -= eps
        args = (lambda x: (x, df.detach())) if t is loc else (lambda x: (loc.detach(), x))
        fd = (float(f(*args(tp))) - float(f(*args(tm)))) / (2 * eps)
        assert abs(fd - float(t.grad[idx])) < 1e-6 * max(1.0, abs(fd))


@pytest.mark.parametrize('trig', ['fast', 'mixed', 'precise', 'strict'])
@pytest.mark.parametrize('nC', [1, 2, 8])
def test_fp32_policies_agree_with_oracle(dev, trig, nC):
    """The fp32 arithmetic policies on a ragged problem (nT = 203: short enough for fp32 to meet the north_star's flat 1e-5),
    single coil (packed kernels), 2 coils (packed kernels, FMA field) and 8 coils (tensor-core forward, weighted reduce)."""
    from mrphy import _ops
    from oracle import bloch_oracle as orc
    p = _random_problem(55 + nC, 2, 333, 203, nC, has_b1=True, relax=True, dtype=f32)
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'],
                                 T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    g = {('in_' + k): v.numpy() for k, v in p.items() if v is not None}
    _ops.set_trig_policy(trig)
    try:
        Mo, gM0, grf, ggr = run_fused(g, dev, f32, p['w'].numpy())
    finally:
        _ops.set_trig_policy(None)
    tol = 3e-5 if trig == 'fast' else ATOL32      # 'mixed' runs the precise forward: same M
    assert Mo.dtype == f32 and grf.dtype == f32
    assert mx(Mo, ref['Mo']) < tol
    assert rel(grf, ref['grf']) < RTOL_G32 and rel(ggr, ref['ggr']) < RTOL_G32 and rel(gM0, ref['gM0']) < RTOL_G32
    if trig == 'strict':
        assert mx(Mo, ref['Mo']) < 2e-7 and rel(grf, ref['grf']) < 1e-6


def test_large_angle_steps_fp32(dev):
    """|b| far beyond the 2 pi range of the half-angle polynomials (phi up to ~1e3 rad per step): the reduce-by-pi path
    (exact to < 1e-8 rad only for phi < ~200, csrc/bloch_math.cuh) must still track the fp64 oracle to fp32's own limit for
    such angles, ~phi * 6e-8 per step."""
    from oracle import bloch_oracle as orc
    p = _random_problem(91, 1, 257, 64, 1, has_b1=True, relax=True, dtype=f32)
    for scale, tol in ((30.0, 2e-4), (400.0, 3e-3)):            # phi_max ~ 0.107 * 36 * 2 * scale ... rad per step
        q = dict(p, gr=p['gr'] * scale)
        ref = orc.applypulse_fwd_bwd(q['M0'], q['rf'], q['gr'], q['loc'], q['w'], df=q['df'], b1=q['b1'], T1=q['T1'],
                                     T2=q['T2'], gamma=q['gam'], dt=q['dt'])
        ref32 = orc.applypulse_fwd_bwd(*(q[k].to(f32) for k in ('M0', 'rf', 'gr', 'loc', 'w')), df=q['df'].to(f32),
                                       b1=q['b1'].to(f32), T1=q['T1'].to(f32), T2=q['T2'].to(f32), gamma=q['gam'].to(f32),
                                       dt=q['dt'].to(f32), dtype=f32)
        g = {('in_' + k): v.numpy() for k, v in q.items() if v is not None}
        Mo, _, _, _ = run_fused(g, dev, f32, q['w'].numpy())
        d, floor = mx(Mo, ref['Mo']), mx(ref32['Mo'], ref['Mo'])
        print(f'[large angles x{scale:g}] max|dM|={d:.2e} (reference algorithm in fp32: {floor:.2e})')
        assert d < max(tol, 1.5 * floor)
        Mo64, _, _, _ = run_fused(g, dev, f64, q['w'].numpy())
        assert mx(Mo64, ref['Mo']) < 1e-10


def test_mixed_small_and_large_angle_tiles(dev):
    """Spins sorted by radius and two batch entries with gradients 30x apart: spin tiles whose steps all stay inside the
    half-angle polynomials' range, tiles that take the large-angle path on most steps, and tiles that mix both inside one
    warp (phi from ~0 to ~25 rad per step), all in one launch; everything must track the fp64 oracle like the reference
    algorithm run in fp32."""
    from oracle import bloch_oracle as orc
    p = _random_problem(77, 2, 3001, 130, 1, has_b1=True, relax=True, dtype=f32)
    order = torch.argsort(p['loc'].norm(dim=-1), dim=1)
    for k in ('loc', 'df', 'M0', 'gam', 'T1', 'T2', 'w', 'b1'):
        idx = order.reshape(order.shape + (1,) * (p[k].dim() - 2)).expand_as(p[k])
        p[k] = torch.gather(p[k], 1, idx)
    p['loc'] = p['loc'] * torch.linspace(0.02, 1.0, 3001, dtype=f64)[None, :, None]
    p['gr'] = p['gr'] * tensor([3.0, 0.1], dtype=f64)[:, None, None]
    p['df'][1] *= 0.05
    ref = orc.applypulse_fwd_bwd(p['M0'], p['rf'], p['gr'], p['loc'], p['w'], df=p['df'], b1=p['b1'], T1=p['T1'],
                                 T2=p['T2'], gamma=p['gam'], dt=p['dt'])
    p32 = {k: v.to(f32) for k, v in p.items()}
    ref32 = orc.applypulse_fwd_bwd(p32['M0'], p32['rf'], p32['gr'], p32['loc'], p32['w'], df=p32['df'], b1=p32['b1'],
                                   T1=p32['T1'], T2=p32['T2'], gamma=p32['gam'], dt=p32['dt'], dtype=f32)
    g = {('in_' + k): v.numpy() for k, v in p.items()}
    for K in (16, 64):
        Mo, gM0, grf, ggr = run_fused(g, dev, f32, p['w'].numpy(), ckpt=K)
        dM, floor = mx(Mo, ref['Mo']), mx(ref32['Mo'], ref['Mo'])
        print(f'[mixed angle tiles K={K}] max|dM|={dM:.2e} (reference fp32 {floor:.2e}) grf {rel(grf, ref["grf"]):.2e} '
              f'ggr {rel(ggr, ref["ggr"]):.2e} gM0 {rel(gM0, ref["gM0"]):.2e}')
        assert dM < _fp32_bound(ref32['Mo'], ref['Mo'])
        assert rel(grf, ref['grf']) < RTOL_G32 and rel(ggr, ref['ggr']) < RTOL_G32 and rel(gM0, ref['gM0']) < RTOL_G32


# ---- SURVEY 8f-2 / f-4: re-parametrisation chain and mask plumbing as single launches -------------------------
@pytest.mark.parametrize('tag', ['sc', 'mc'])
@pytest.mark.parametrize('dtype', [f64, f32])
def test_design_waveform_kernel_matches_reference(dev, golden, tag, dtype):
    """utils.tρθ2rf / lρθ2rf / ts2s / s2g / ts2g / tρθts2rfgr on CUDA tensors (one launch each way, csrc/design_ops.cu)
    against the unmodified reference's outputs and autograd gradients and against the numpy oracle.
    Tolerance: fp64 1e-12 relative; fp32 2e-6 relative to the largest value (inputs rounded to fp32, arithmetic in
    double with one final rounding; the fp32 running sum of the reference itself differs by ~1e-6)."""
    from mrphy import utils, _cabi
    from oracle import bloch_oracle as orc
    g = {k[len(tag) + 1:]: v for k, v in golden('reparam').items() if k.startswith(tag + '_')}
    tol = 1e-12 if dtype == f64 else 2e-6
    t = {k: T(v, dev, dtype) for k, v in g.items()}
    near = lambda a, b: mx(a, b) <= tol * float(np.abs(b).max())
    rho, theta, ts = (t[k].clone().requires_grad_(True) for k in ('rho', 'theta', 'ts'))
    n0 = _cabi.launch_counter
    for kind, fn, logit in (('t', utils.tρθ2rf, False), ('l', utils.lρθ2rf, True)):
        rf = fn(rho, theta, t['rfmax'])
        assert rf.dtype == dtype and near(rf, g['rf_' + kind])
        grho, gtheta = torch.autograd.grad((rf * t['wrf']).sum(), (rho, theta))
        assert near(grho, g['grho_' + kind]) and near(gtheta, g['gtheta_' + kind])
        o_rf = orc.reparam_fwd(rho.detach().cpu().numpy(), theta.detach().cpu().numpy(), t['rfmax'].cpu().numpy(),
                               ts.detach().cpu().numpy(), t['smax'].cpu().numpy(), t['dt'].cpu().numpy(), logit=logit)[0]
        assert mx(rf, o_rf) <= (1e-13 if dtype == f64 else 1e-7) * float(np.abs(o_rf).max())   # same (rounded) inputs
    assert _cabi.launch_counter - n0 == 4          # two forwards + two adjoints, one launch each
    s = utils.ts2s(ts, t['smax'])
    gr = utils.s2g(s, t['dt'])
    assert near(s, g['s']) and near(gr, g['gr'])
    gts_s, = torch.autograd.grad((s * t['wg']).sum(), (ts,), retain_graph=True)
    assert near(gts_s, g['gts_s'])
    gts, = torch.autograd.grad((gr * t['wg']).sum(), (ts,))
    assert near(gts, g['gts'])
    assert near(utils.ts2g(ts, t['smax'], t['dt']), g['gr'])
    n0 = _cabi.launch_counter
    rf2, gr2 = utils.tρθts2rfgr(rho, theta, ts, t['rfmax'], t['smax'], t['dt'])
    ((rf2 * t['wrf']).sum() + (gr2 * t['wg']).sum()).backward()
    assert _cabi.launch_counter - n0 == 2          # the whole chain: ONE launch forward, ONE backward
    assert near(rf2, g['rf_t']) and near(gr2, g['gr'])
    assert near(rho.grad, g['grho_t']) and near(theta.grad, g['gtheta_t']) and near(ts.grad, g['gts'])


def test_design_waveform_long_and_scalar_constants(dev):
    """nT = 4001 (16 chunks of the running sum, ragged tail), scalar rfmax / smax / default fp64 dt0 like upstream's
    defaults, against the torch expressions the reference is made of; and the cases the kernel leaves to torch."""
    from mrphy import utils, dt0, rfmax0, smax0, π
    gen = torch.Generator().manual_seed(5)
    N, nT = 3, 4001
    rho, theta, ts = (torch.randn((N, c, nT), generator=gen, dtype=f64).to(dev) for c in (1, 1, 3))
    rf, gr = utils.tρθts2rfgr(rho, theta, ts, rfmax0, smax0)
    rf_ref = rho.atan() / π * 2 * rfmax0.to(dev) * torch.cat((theta.cos(), theta.sin()), dim=1)
    gr_ref = dt0.to(dev) * torch.cumsum(ts.atan() / π * 2 * smax0.to(dev), dim=2)
    assert rel(rf, rf_ref) < 1e-14 and rel(gr, gr_ref) < 1e-13
    # per-axis 1-D smax, per-pulse dt
    smax = tensor([1e3, 2e3, 3e3], dtype=f64, device=dev)
    dtn = tensor([4e-6, 2e-6, 1e-5], dtype=f64, device=dev)
    g2 = utils.ts2g(ts, smax, dtn)
    g2_ref = dtn[:, None, None] * torch.cumsum(ts.atan() / π * 2 * smax[..., None], dim=2)
    assert rel(g2, g2_ref) < 1e-13
    # gradients w.r.t. the constants are not the kernel's business: torch expression, same numbers
    smax_g = smax.clone().requires_grad_(True)
    s = utils.ts2s(ts, smax_g)
    s.sum().backward()
    assert smax_g.grad is not None and rel(s, ts.atan() / π * 2 * smax[..., None]) < 1e-15


@pytest.mark.parametrize('dtype', [f64, f32])
def test_mask_kernel_embed_extract(dev, golden, dtype):
    """SpinArray.embed / extract through the one-pass gather kernel: bit-exact against the reference's outputs (NaN
    pattern included) and differentiable (transposed map)."""
    from mrphy import mobjs, _cabi
    g = golden('reparam')
    sa = mobjs.SpinArray((2, 5, 4, 3), mask=tensor(g['mask']).to(dev), dtype=dtype, device=dev)
    v_ = T(g['mask_v_'], dev, dtype).requires_grad_(True)
    n0 = _cabi.launch_counter
    emb = sa.embed(v_)
    assert _cabi.launch_counter == n0 + 1
    want = tensor(g['mask_embedded']).to(dtype).numpy()
    got = emb.detach().cpu().numpy()
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.array_equal(np.nan_to_num(got), np.nan_to_num(want))
    w = torch.randn(emb.shape, device=dev, dtype=dtype)
    torch.nan_to_num(emb * w).sum().backward()
    assert torch.equal(v_.grad, sa.extract(w))
    full = T(g['mask_full'], dev, dtype).requires_grad_(True)
    ex = sa.extract(full)
    assert np.array_equal(ex.detach().cpu().numpy(), tensor(g['mask_extracted']).to(dtype).numpy())
    w2 = torch.randn(ex.shape, device=dev, dtype=dtype)
    (ex * w2).sum().backward()
    assert torch.equal(full.grad, torch.nan_to_num(sa.embed(w2)))
    # a full-size cube: 64^3 with a spherical mask, round trip
    n = 64
    ax = torch.arange(n, device=dev) - n // 2
    mask = ((ax[:, None, None] ** 2 + ax[None, :, None] ** 2 + ax[None, None, :] ** 2) < (n // 2) ** 2)[None]
    big = mobjs.SpinArray((1, n, n, n), mask=mask, dtype=dtype, device=dev)
    m_ = torch.randn((1, big.nM, 3), device=dev, dtype=dtype)
    e = big.embed(m_)
    assert torch.equal(big.extract(e), m_) and bool(torch.isnan(e[~mask.expand(1, n, n, n)]).all())


def test_design_loop_with_fresh_pulses_has_no_host_sync(dev):
    """Every design iteration builds a NEW Pulse from the optimiser's variables (so `dt` is a new device tensor each time):
    after the first iteration nothing on the path may read the device (checkpoint policy, mask indices, constants) --
    `torch.cuda.set_sync_debug_mode('error')` turns any synchronising call into an exception."""
    from mrphy import mobjs, utils, rfmax0, smax0
    kw = {'dtype': f32, 'device': dev}
    n, nT = 12, 96
    gen = torch.Generator().manual_seed(3)
    ax = torch.arange(n) - n // 2
    mask = ((ax[:, None, None] ** 2 + ax[None, :, None] ** 2 + ax[None, None, :] ** 2) < (n // 2) ** 2)[None].to(dev)
    cube = mobjs.SpinCube((1, n, n, n), tensor([[24., 24., 24.]]), mask=mask, **kw)
    v = [(torch.randn((1, c, nT), generator=gen) * 0.3).to(**kw).requires_grad_(True) for c in (1, 1, 3)]
    tgt = tensor([0., 1., 0.], **kw)

    def iteration():
        rf, gr = utils.tρθts2rfgr(v[0], v[1], v[2], rfmax0, smax0)
        M = cube.applypulse(mobjs.Pulse(rf=rf, gr=gr, **kw), doEmbed=True)
        loss = ((cube.extract(M) - tgt) ** 2).sum()
        for x in v:
            x.grad = None
        loss.backward()
        return loss

    first = iteration()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        for _ in range(3):
            again = iteration()
    finally:
        torch.cuda.set_sync_debug_mode('default')
    assert torch.equal(first, again) and all(x.grad is not None and bool(torch.isfinite(x.grad).all()) for x in v)
    # ... which is what lets the WHOLE iteration (re-parametrisation, fresh Pulse, mask kernels, simulation, adjoint) record
    # into one CUDA graph; a replay after an in-place update of the variables equals the eager iteration bit for bit
    from mrphy import graphs
    eager_grads = [x.grad.clone() for x in v]
    del first, again
    captured = graphs.capture(iteration, params=v)
    captured.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(x.grad, g) for x, g in zip(v, eager_grads))
    with torch.no_grad():
        for x in v:
            x.mul_(0.9)
    captured.replay()
    replayed = [x.grad.clone() for x in v]
    iteration()
    assert all(torch.equal(x.grad, g) for x, g in zip(v, replayed))


@pytest.mark.parametrize('dtype', [f32, f64])
def test_gradient_rows_on_demand(dev, dtype):
    """When only rf (an RF-only design on a fixed trajectory) or only gr needs a gradient, the backward neither forms nor
    reduces the other rows (flags MRPHY_SKIP_GRF / MRPHY_SKIP_GGR): the gradients that ARE asked for must be bitwise
    those of the full backward, the others None -- on the default kernels (big enough for the SM-aware grid) and on a
    multi-coil problem (generic kernels: rows skipped in the finalize only)."""
    from mrphy import _ops
    gen = torch.Generator().manual_seed(9)
    U = lambda *s: (torch.rand(s, generator=gen, dtype=f64) * 2 - 1)
    for N, nM, nT, nC in ((1, 148 * 4 * 256 + 77, 130, 0), (2, 300, 97, 2), (1, 517, 70, 8)):
        rf = (U(N, 2, nT, nC) if nC else U(N, 2, nT)) * 0.1
        b1 = U(N, nM, 2, max(nC, 1)) * 0.1
        b1[:, :, 0] += 1
        t = lambda x: x.to(dtype).to(dev)
        args = dict(loc_=t(U(N, nM, 3) * 12), Δf_=t(U(N, nM) * 200), b1Map_=t(b1), T1_=t(1.0 + 0.5 * U(N, nM)),
                    T2_=t(0.06 + 0.05 * U(N, nM)), γ_=tensor(4257.6, dtype=f64, device=dev), dt=tensor([4e-6], dtype=f64, device=dev))
        M0, w = t(torch.nn.functional.normalize(U(N, nM, 3), dim=-1)), t(U(N, nM, 3))
        grads = {}
        for which in ('both', 'rf', 'gr', 'M'):
            r = t(rf).requires_grad_(which in ('both', 'rf'))
            g = t(U(N, 3, nT) * 0 + 1.3).requires_grad_(which in ('both', 'gr'))
            m = M0.clone().requires_grad_(which == 'M')
            Mo = _ops.fused_applypulse(m, r, g, **args)
            (Mo * w).sum().backward()
            grads[which] = (r.grad, g.grad, m.grad)
        assert grads['rf'][1] is None and grads['gr'][0] is None and grads['M'][0] is None and grads['M'][1] is None
        assert torch.equal(grads['rf'][0], grads['both'][0]) and torch.equal(grads['gr'][1], grads['both'][1])
        assert grads['M'][2] is not None and bool(torch.isfinite(grads['M'][2]).all())
