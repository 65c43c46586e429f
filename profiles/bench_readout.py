"""The receive signal summed over spins inside the fused kernels (`readout=`) against the same step without it and against
`record=` followed by an einsum over Mt for the same signal.

    python profiles/bench_readout.py [--steps 7] [--warmup 2] [--out profiles/r5_readout.json] [--c5]

C2 (64^3 spins x 1000 steps), fp32, precise policy, relaxation on, 1 and 8 transmit coils with a b1Map; s in {1, 4, 16},
nRx in {1, 8}.  Per case and route (off | readout | record + einsum):
  fwd_ms, bwd_ms   the main forward / backward kernel alone (the library's CUDA events, mrphy_kernel_timing)
  ms               one fwd+bwd step between CUDA events, loss = sum(M*M) + <w, S>
  peak_gb          torch.cuda.max_memory_allocated over the timed steps
--c5 adds C5 (256^3 x 4000, 1 coil, s = 1, nRx = 1), where the record route does not fit on the card: off and readout only.
L2 overwritten (256 MB memset) before every timed step, median of --steps, every shape warmed up first; card name and
power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), 'mrphy.py_b200'))

import torch  # noqa: E402

from mrphy import _cabi, _ops  # noqa: E402

f64 = torch.float64


def problem(nM, nT, nC, nRx, dev):
    g = torch.Generator(device=dev).manual_seed(0)
    U = lambda *s: torch.rand(s, generator=g, device=dev) * 2 - 1
    p = dict(M=torch.nn.functional.normalize(U(1, nM, 3), dim=-1), loc=U(1, nM, 3) * 12, df=U(1, nM) * 100,
             rf=U(1, 2, nT, nC) * 0.02 if nC > 1 else U(1, 2, nT) * 0.1, gr=U(1, 3, nT) * 2,
             b1=U(1, nM, 2, nC) * 0.1 if nC > 1 else U(1, nM, 2) * 0.1, rx=U(1, nM, 2, nRx))
    p['b1'][:, :, 0] += 1
    p['T1'], p['T2'] = torch.ones(1, nM, device=dev), torch.full((1, nM), 0.08, device=dev)
    p['gam'], p['dt'] = torch.tensor(4257.6, dtype=f64, device=dev), torch.tensor([4e-6], dtype=f64, device=dev)
    return p


def signal(Mt, rx):
    mx, my, cx, cy = Mt[..., 0], Mt[..., 1], rx[:, :, 0], rx[:, :, 1]
    return torch.stack([torch.einsum('nik,nir->nrk', cx, mx) - torch.einsum('nik,nir->nrk', cy, my),
                        torch.einsum('nik,nir->nrk', cx, my) + torch.einsum('nik,nir->nrk', cy, mx)], 1)


def step(p, route, s, w, kernel_ms=None):
    """One fwd+bwd step; with `kernel_ms` (a list) also the forward and backward kernel times (synchronises between)."""
    L = _cabi.lib()
    rf, gr = p['rf'].detach().requires_grad_(True), p['gr'].detach().requires_grad_(True)
    kw = dict(Δf_=p['df'], b1Map_=p['b1'], T1_=p['T1'], T2_=p['T2'], γ_=p['gam'], dt=p['dt'])
    if route == 'off':
        M = _ops.fused_applypulse(p['M'], rf, gr, p['loc'], **kw)
        S = None
    elif route == 'readout':
        M, S = _ops.fused_applypulse(p['M'], rf, gr, p['loc'], readout=s, rxMap_=p['rx'], **kw)
    else:
        M, Mt = _ops.fused_applypulse(p['M'], rf, gr, p['loc'], record=s, **kw)
        S = signal(Mt, p['rx'])
    if kernel_ms is not None:
        kernel_ms.append(L.mrphy_last_kernel_ms())
    loss = (M * M).sum() + ((S * w).sum() if S is not None else 0)
    loss.backward()
    if kernel_ms is not None:
        kernel_ms.append(L.mrphy_last_kernel_ms())


def med(x):
    return sorted(x)[len(x) // 2]


def run(p, route, s, w, steps, warmup, flush):
    L = _cabi.lib()
    for _ in range(warmup):
        step(p, route, s, w)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ms = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(p, route, s, w)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    peak = torch.cuda.max_memory_allocated() / 1e9
    fwd, bwd = [], []
    L.mrphy_kernel_timing(1)
    try:
        for _ in range(steps):
            flush.zero_()
            k = []
            step(p, route, s, w, k)
            fwd.append(k[0])
            bwd.append(k[1])
    finally:
        L.mrphy_kernel_timing(0)
    return dict(ms=med(ms), ms_all=ms, fwd_ms=med(fwd), bwd_ms=med(bwd), fwd_all=fwd, bwd_all=bwd, peak_gb=peak)


def case(res, size, nM, nT, nC, nRx, s, routes, a, dev, flush, base):
    p = problem(nM, nT, nC, nRx, dev)
    w = torch.rand(1, 2, nT // s, nRx, device=dev) - 0.5
    out = {}
    for route in routes:
        r = run(p, route, s, w, a.steps, a.warmup, flush)
        row = dict(size=size, nM=nM, nT=nT, nC=nC, nRx=nRx, s=s, route=route, **r)
        if base is not None:
            row.update(step_over_off=r['ms'] / base['ms'], fwd_over_off=r['fwd_ms'] / base['fwd_ms'],
                       bwd_over_off=r['bwd_ms'] / base['bwd_ms'], peak_over_off_gb=r['peak_gb'] - base['peak_gb'])
        out[route] = row
    if 'record' in out and 'readout' in out:
        out['readout']['record_over_readout'] = out['record']['ms'] / out['readout']['ms']
    for row in out.values():
        print(json.dumps({k: v for k, v in row.items() if not k.endswith('_all')}), flush=True)
        res['results'].append(row)
    del p
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=7)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=os.path.join(HERE, 'r5_readout.json'))
    ap.add_argument('--c5', action='store_true')
    a = ap.parse_args()
    if a.steps < 5:
        raise SystemExit('--steps must be at least 5 (the median of fewer is noise)')
    dev = torch.device('cuda:0')
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({'gpu': smi}), flush=True)
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    res = dict(gpu=smi, torch=torch.__version__, steps=a.steps, warmup=a.warmup, policy=_ops.trig_policy(), results=[])
    nM, nT = 64 ** 3, 1000
    for nC in (1, 8):
        base = case(res, 'C2', nM, nT, nC, 1, 1, ('off',), a, dev, flush, None)['off']
        for s in (1, 4, 16):
            for nRx in (1, 8):
                case(res, 'C2', nM, nT, nC, nRx, s, ('readout', 'record'), a, dev, flush, base)
    if a.c5:
        base = case(res, 'C5', 256 ** 3, 4000, 1, 1, 1, ('off',), a, dev, flush, None)['off']
        case(res, 'C5', 256 ** 3, 4000, 1, 1, 1, ('readout',), a, dev, flush, base)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
