"""Per-spin (B0 / B1 map) gradients: cost of one fwd+bwd step on the fused path against rf/gr gradients only and against the
explicit-field route.

    python profiles/bench_spin_grads.py [--steps 5] [--warmup 2] [--out profiles/r3_spin_grads.json]

Cases, fp32, precise policy:
  a  rf/gr gradients only (the design step)
  b  rf/gr + Δf_ + b1Map_ gradients (fused backward with per-spin sums)
  c  Δf_ + b1Map_ only, fixed pulse (no spin reduction, no finalize)
  d  the explicit-field route for the gradients of b: sims.blochsim(M, rfgr2beff(...)) -- skipped at C5, where the dense
     field and its gradient would need 2 x 805 GB
at C2 (64^3 x 1000; 1 and 8 coils) and C5 (256^3 x 4000; 1 coil).  CUDA events around each step, L2 overwritten (256 MB
memset) before every step, peak torch.cuda.max_memory_allocated per case; card name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), 'mrphy.py_b200'))

import torch  # noqa: E402

from mrphy import _ops, beffective, sims  # noqa: E402

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


def step(p, case):
    wave = case in 'abd'
    spin = case in 'bcd'
    rf, gr = p['rf'].detach().requires_grad_(wave), p['gr'].detach().requires_grad_(wave)
    df, b1 = p['df'].detach().requires_grad_(spin), p['b1'].detach().requires_grad_(spin)
    if case == 'd':
        B = beffective.rfgr2beff(rf, gr, p['loc'], Δf=df, b1Map=b1, γ=p['gam'])
        Mo = sims.blochsim(p['M'], B, T1=p['T1'], T2=p['T2'], γ=p['gam'], dt=p['dt'])
    else:
        Mo = _ops.fused_applypulse(p['M'], rf, gr, p['loc'], Δf_=df, b1Map_=b1, T1_=p['T1'], T2_=p['T2'], γ_=p['gam'],
                                   dt=p['dt'])
    (Mo * Mo).sum().backward()


def run(p, case, steps, warmup, flush):
    for _ in range(warmup):
        step(p, case)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ms = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        step(p, case)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return dict(ms=sorted(ms)[len(ms) // 2], ms_all=ms, peak_gb=torch.cuda.max_memory_allocated() / 1e9)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--out', default=os.path.join(HERE, 'r3_spin_grads.json'))
    ap.add_argument('--sizes', default='C2x1,C2x8,C5x1')
    a = ap.parse_args()
    dev = torch.device('cuda:0')
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    res = dict(gpu=smi, torch=torch.__version__, steps=a.steps, warmup=a.warmup, policy=_ops.trig_policy(), results=[])
    sizes = dict(C2=(64 ** 3, 1000), C5=(256 ** 3, 4000))
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    for tag in a.sizes.split(','):
        name, nC = tag.split('x')
        nM, nT = sizes[name]
        p = problem(nM, nT, int(nC), dev)
        for case in 'abcd':
            row = dict(size=name, nM=nM, nT=nT, nC=int(nC), case=case)
            if case == 'd' and name == 'C5':
                row['skipped'] = 'dense Beff and dL/dBeff need 2 x %.0f GB' % (nM * nT * 12 / 1e9)
            else:
                r = run(p, case, a.steps, a.warmup, flush)
                row.update(r, spin_steps_per_s=nM * nT / (r['ms'] * 1e-3))
            print(json.dumps(row), flush=True)
            res['results'].append(row)
        del p
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps({'gpu': smi}))


if __name__ == '__main__':
    main()
