"""Recording the magnetisation every s steps (`record=`): kernel time, step time and peak memory against the same step
without recording.

    python profiles/bench_record.py [--steps 7] [--warmup 2] [--out profiles/r4_record.json]

C2 (64^3 spins x 1000 steps), fp32, precise policy, relaxation on, 1 coil and 8 coils with a b1Map; record in {off, 1, 4,
16, 250}.  Per case:
  fwd_ms, bwd_ms   the main forward / backward kernel alone (the library's CUDA events, mrphy_kernel_timing), with the
                   loss on Mt and on M (off: on M)
  ms               one fwd+bwd step between CUDA events, loss = sum(M*M) + sum(Mt*Mt)
  peak_gb          torch.cuda.max_memory_allocated over the timed steps
  mt_write_tb_s    Mt bytes written (nM * nR * 3 * 4) / fwd_ms, next to the copy bandwidth measured in the same run
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


def problem(nM, nT, nC, dev):
    g = torch.Generator(device=dev).manual_seed(0)
    U = lambda *s: torch.rand(s, generator=g, device=dev) * 2 - 1
    p = dict(M=torch.nn.functional.normalize(U(1, nM, 3), dim=-1), loc=U(1, nM, 3) * 12, df=U(1, nM) * 100,
             rf=U(1, 2, nT, nC) * 0.02 if nC > 1 else U(1, 2, nT) * 0.1, gr=U(1, 3, nT) * 2,
             b1=U(1, nM, 2, nC) * 0.1 if nC > 1 else U(1, nM, 2) * 0.1)
    p['b1'][:, :, 0] += 1
    p['T1'], p['T2'] = torch.ones(1, nM, device=dev), torch.full((1, nM), 0.08, device=dev)
    p['gam'], p['dt'] = torch.tensor(4257.6, dtype=f64, device=dev), torch.tensor([4e-6], dtype=f64, device=dev)
    return p


def step(p, record, kernel_ms=None):
    """One fwd+bwd step; with `kernel_ms` (a list) also the forward and backward kernel times (synchronises between)."""
    L = _cabi.lib()
    rf, gr = p['rf'].detach().requires_grad_(True), p['gr'].detach().requires_grad_(True)
    out = _ops.fused_applypulse(p['M'], rf, gr, p['loc'], Δf_=p['df'], b1Map_=p['b1'], T1_=p['T1'], T2_=p['T2'],
                                γ_=p['gam'], dt=p['dt'], record=record)
    if kernel_ms is not None:
        kernel_ms.append(L.mrphy_last_kernel_ms())
    if record is None:
        loss = (out * out).sum()
    else:
        Mo, Mt = out
        loss = (Mo * Mo).sum() + (Mt * Mt).sum()
    loss.backward()
    if kernel_ms is not None:
        kernel_ms.append(L.mrphy_last_kernel_ms())


def med(x):
    return sorted(x)[len(x) // 2]


def run(p, record, steps, warmup, flush):
    L = _cabi.lib()
    for _ in range(warmup):
        step(p, record)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ms = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(p, record)
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
            step(p, record, k)
            fwd.append(k[0])
            bwd.append(k[1])
    finally:
        L.mrphy_kernel_timing(0)
    return dict(ms=med(ms), ms_all=ms, fwd_ms=med(fwd), bwd_ms=med(bwd), fwd_all=fwd, bwd_all=bwd, peak_gb=peak)


def copy_bandwidth(dev, flush, reps=9):
    """dst.copy_(src) of 2 GiB: (bytes read + bytes written) / time, median."""
    n = 2 ** 31
    src, dst = torch.empty(n, dtype=torch.uint8, device=dev), torch.empty(n, dtype=torch.uint8, device=dev)
    src.fill_(1)
    dst.copy_(src)
    out = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dst.copy_(src)
        e1.record()
        torch.cuda.synchronize()
        out.append(2 * n / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    del src, dst
    torch.cuda.empty_cache()
    return med(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=7)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=os.path.join(HERE, 'r4_record.json'))
    ap.add_argument('--coils', default='1,8')
    ap.add_argument('--records', default='off,1,4,16,250')
    a = ap.parse_args()
    if a.steps < 5:
        raise SystemExit('--steps must be at least 5 (the median of fewer is noise)')
    dev = torch.device('cuda:0')
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({'gpu': smi}), flush=True)
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    copy_tb_s = copy_bandwidth(dev, flush)
    res = dict(gpu=smi, torch=torch.__version__, steps=a.steps, warmup=a.warmup, policy=_ops.trig_policy(),
               copy_tb_s=copy_tb_s, results=[])
    print(json.dumps({'copy_tb_s': copy_tb_s}), flush=True)
    nM, nT = 64 ** 3, 1000
    for nC in (int(c) for c in a.coils.split(',')):
        p = problem(nM, nT, nC, dev)
        base = None
        for rec in a.records.split(','):
            record = None if rec == 'off' else int(rec)
            r = run(p, record, a.steps, a.warmup, flush)
            row = dict(size='C2', nM=nM, nT=nT, nC=nC, record=rec, **r)
            if record is None:
                base = row
            else:
                mt_bytes = nM * (nT // record) * 3 * 4
                row.update(mt_gb=mt_bytes / 1e9, mt_write_tb_s=mt_bytes / (r['fwd_ms'] * 1e-3) / 1e12,
                           mt_write_over_copy=mt_bytes / (r['fwd_ms'] * 1e-3) / 1e12 / copy_tb_s)
                if base is not None:
                    row.update(step_over_off=r['ms'] / base['ms'], fwd_over_off=r['fwd_ms'] / base['fwd_ms'],
                               bwd_over_off=r['bwd_ms'] / base['bwd_ms'])
            print(json.dumps({k: v for k, v in row.items() if not k.endswith('_all')}), flush=True)
            res['results'].append(row)
        del p
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
