#!/usr/bin/env python
"""bench.py -- spin·steps/s of the fused Bloch simulation, forward + adjoint backward.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload c2|c3|c4|c5|small]
                    [--dtype f32|f64] [--scaling strong|weak] [--no-graph] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input (BASELINE.md / SURVEY.md 8d):
``M = spins.applypulse(pulse, loc_=..., Δf_=..., b1Map_=...)``; ``loss = ((M - target)**2).sum()``; ``loss.backward()``
giving ``pulse.rf.grad``, ``pulse.gr.grad`` (+ ONE in-place NCCL all-reduce of the flat gradient buffer when N > 1).

Default workload = the north_star design problem, BASELINE config C5: SpinCube 256^3 (16.7 M spins), nT = 4000, dt = 4 us,
fp32, STRONG scaling -- the same global cube at every N, cut into contiguous compact-spin slabs by
``mrphy.parallel.shard_spins`` (at N = 1 the whole cube runs on one GPU: 13 GB of checkpoints).  C2 (64^3 x 1000, the
1-GPU configuration of BASELINE.json) is measured in the same run and reported under ``"c2"``.

Prints ONE JSON line (rank 0).  ``value`` is measured with inputs resident in HBM (CUDA events around each step, L2
flushed between steps; the whole step INCLUDING the all-reduce is replayed from a CUDA graph unless --no-graph);
``e2e`` goes through the same public API eagerly but copies every input from pinned host memory every step and reads the
loss and gradients back into pinned memory, all inside one wall-clock timed region of K steps.
``--impl reference`` times the UNMODIFIED reference (oracle/_ref, staged by oracle/Makefile: its own
``SpinCube.applypulse`` + ``backward`` through its own public API) on the host cores, on a bounded sub-cube of the same
workload; without a staged copy it times the oracle port and says so (``cpu_baseline.kind``).

``--dump-outputs DIR`` writes what the last timed step returned (M, rf.grad, gr.grad, loss) as ``DIR/<name>.npy``.  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True        # the tree may be read-only: importing the package from it must not write there

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = 'spin_steps_per_sec_fwd_bwd'
UNIT = 'spin·steps/s'
FLOP_PER_SPIN_STEP = 223.0        # SURVEY.md 8(d): fwd 62 + bwd 161 algorithmic flop (fp32, 1 coil, relax, b1, df)
FLOP_FWD, FLOP_BWD = 62.0, 161.0
ISSUE_SLOTS = 151.0               # SURVEY.md 8(d): 145 FP32-pipe instructions + 6 MUFU per spin-step, fwd + bwd
WORKLOADS = {   # name: (N, n, nT)
    'c2': (1, 64, 1000), 'c3': (1, 128, 2000), 'c4': (64, 40, 1000), 'c5': (1, 256, 4000), 'small': (1, 16, 200),
}


def use_ours():
    for p in (ROOT, os.path.join(ROOT, 'mrphy.py_b200')):
        if p not in sys.path:
            sys.path.insert(0, p)


def use_reference():
    """-> 'reference' with oracle/_ref (the unmodified reference) importable as `mrphy`, else 'port'."""
    ref = os.path.join(ROOT, 'oracle', '_ref')
    if os.path.isdir(os.path.join(ref, 'mrphy')):
        sys.path[:] = [p for p in sys.path if os.path.abspath(p or '.') != os.path.join(ROOT, 'mrphy.py_b200')]
        sys.path.insert(0, ref)
        return 'reference'
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    return 'port'


def peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            mp = json.load(f)
        return float(mp['hbm_gbs']), float(mp['sm_max_mhz']), 'measured'
    except Exception:
        return 6650.0, 1965.0, 'fallback'


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace('.', '').isdigit()]
        mxs = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace('.', '').isdigit()]
        pw = [float(r[3]) for r in self.rows if len(r) >= 9 and r[3].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows if len(r) >= 9 for n, v in zip(names, r[5:9]) if v.lower() == 'active'})
        busy = [s for s, p in zip(sm, pw) if p > 0.5 * max(pw)] if pw and len(pw) == len(sm) else sm
        return {'sm_mhz': float(np.median(busy)) if busy else None, 'sm_max_mhz': max(mxs) if mxs else None,
                'reasons': reasons, 'samples': len(sm), 'power_w_max': max(pw) if pw else None}


def synth(N, n_x, n, nT, dtype, seed=0, x_off=0, n_x_total=None, interp=1, mobjs=None):
    """Seeded synthetic slab (SURVEY 8d distributions), generated in fp64 then rounded to `dtype`.
    Slab = x-indices [x_off, x_off+n_x) of a (n_x_total, n, n) grid with 24 cm fov per 64 voxels... of an n-voxel axis.
    interp > 1 (BASELINE config C3, "multi-scale interpT design"): the waveform is drawn with nT/interp samples at
    interp*4 us in fp64 and brought to nT samples at 4 us by `Pulse.interpT` (SURVEY 8d: fp64, or the grid is 1 short)."""
    n_x_total = n_x if n_x_total is None else n_x_total
    gen = torch.Generator().manual_seed(seed + 1000 * x_off)
    U = lambda *s: torch.rand(s, generator=gen, dtype=torch.float64) * 2 - 1
    fov = torch.tensor([24.0 * n_x_total / n, 24.0, 24.0], dtype=torch.float64)
    ax = [(torch.arange(x_off, x_off + n_x, dtype=torch.float64) - n_x_total // 2) / n_x_total,
          (torch.arange(n, dtype=torch.float64) - n // 2) / n, (torch.arange(n, dtype=torch.float64) - n // 2) / n]
    g = torch.meshgrid(*ax, indexing='ij')
    loc = torch.stack([fov[i] * g[i].reshape(-1) for i in range(3)], dim=-1)[None].expand(N, -1, 3).contiguous()
    nM = loc.shape[1]
    wgen = torch.Generator().manual_seed(seed)          # the waveform is the same on every rank
    W = lambda *s: torch.rand(s, generator=wgen, dtype=torch.float64) * 2 - 1
    if interp > 1:
        if mobjs is None:
            from mrphy import mobjs
        assert nT % interp == 0
        f8 = torch.float64
        coarse = mobjs.Pulse(rf=W(N, 2, nT // interp) * 0.1, gr=W(N, 3, nT // interp) * 2,
                             dt=torch.tensor(4e-6 * interp, dtype=f8), dtype=f8)
        fine = coarse.interpT(dt=torch.tensor(4e-6, dtype=f8))
        rf, gr = fine.rf, fine.gr
        assert rf.shape[2] == nT, rf.shape
    else:
        rf, gr = W(N, 2, nT) * 0.1, W(N, 3, nT) * 2
    df = U(N, nM) * 200
    b1 = U(N, nM, 2) * 0.1
    b1[:, :, 0] += 1
    M0 = torch.tensor([0., 0., 1.], dtype=torch.float64).expand(N, nM, 3).contiguous()
    return {k: v.to(dtype) for k, v in dict(rf=rf, gr=gr, loc=loc, df=df, b1=b1, M0=M0).items()}


def workload_desc(workload, scaling, world):
    N, n, nT = WORKLOADS[workload]
    return (f'{workload.upper()}: SpinCube {n}^3 x N={N} ' +
            ('per GPU' if scaling == 'weak' else f'split over {world} GPU{"s" if world > 1 else ""} (mrphy.parallel.shard_spins)') +
            f', nT={nT}, dt=4us' + (f' (Pulse.interpT from {nT // 5} x 20us)' if workload == 'c3' else '') +
            ', b1Map+df+relaxation, fwd+adjoint bwd')


def pick_scaling(args):
    return args.scaling or ('strong' if args.workload == 'c5' else 'weak')


# ======================================================================================================================
# our arm
class Problem:
    """One workload on this rank: the rank's slab of spins (through mrphy.parallel.shard_spins for strong scaling), the
    replicated pulse, and the step."""

    def __init__(self, workload, scaling, dtype, dev, rank, world):
        from mrphy import mobjs, parallel
        self.parallel = parallel
        self.keep_M, self.M = False, None     # keep_M: hold on to the magnetisation of the latest step in self.M
        self.N, self.n, self.nT = WORKLOADS[workload]
        N, n, nT = self.N, self.n, self.nT
        self.dtype, self.dev, self.world = dtype, dev, world
        kw = {'dtype': dtype, 'device': dev}
        itp = 5 if workload == 'c3' else 1     # C3: the pulse comes out of Pulse.interpT (400 x 20 us -> 2000 x 4 us)
        if scaling == 'strong':
            # the SAME global cube at every world size; the shipped helper cuts this rank's contiguous compact-spin slab
            glob = synth(N, n, n, nT, dtype, interp=itp)
            cpu = {'dtype': dtype, 'device': torch.device('cpu')}
            sp_g = mobjs.SpinArray((N, n ** 3), M_=glob['M0'], **cpu)
            sp, skw = parallel.shard_spins(sp_g, rank, world, loc_=glob['loc'], Δf_=glob['df'], b1Map_=glob['b1'], device=dev)
            lo, hi = parallel.shard_range(n ** 3, rank, world)
            host = dict(rf=glob['rf'], gr=glob['gr'], loc=glob['loc'][:, lo:hi].contiguous(), df=glob['df'][:, lo:hi].contiguous(),
                        b1=glob['b1'][:, lo:hi].contiguous(), M0=glob['M0'][:, lo:hi].contiguous())
            del sp_g
        else:                             # weak: every rank owns an n^3 slab of an (n*world) x n x n cube
            host = synth(N, n, n, nT, dtype, x_off=rank * n, n_x_total=n * world, interp=itp)
        self.host = host
        self.nM = host['loc'].shape[1]
        self.tgt = torch.tensor([0., 1., 0.], **kw)
        if scaling == 'strong':          # the objects the timed region runs on are the ones mrphy.parallel.shard_spins built
            self.sp = sp
            self.d = {'loc': skw['loc_'], 'df': skw['Δf_'], 'b1': skw['b1Map_']}
            self.pulse = mobjs.Pulse(rf=glob['rf'].to(dev).requires_grad_(True), gr=glob['gr'].to(dev).requires_grad_(True), **kw)
            assert self.sp.nM == self.nM and self.d['loc'].shape == (N, self.nM, 3)
        else:
            self.sp, self.pulse, self.d = self.make_objects(host)
        self.units_local = float(N) * self.nM * nT

    def make_objects(self, src, non_blocking=False):
        from mrphy import mobjs
        kw = {'dtype': self.dtype, 'device': self.dev}
        d = {k: v.to(self.dev, non_blocking=non_blocking) for k, v in src.items()}
        sp = mobjs.SpinArray((self.N, self.nM), M_=d['M0'], **kw)
        pulse = mobjs.Pulse(rf=d['rf'].requires_grad_(True), gr=d['gr'].requires_grad_(True), **kw)
        return sp, pulse, d

    def local_step(self, sp=None, pulse=None, d=None):
        sp, pulse, d = (self.sp, self.pulse, self.d) if sp is None else (sp, pulse, d)
        M = sp.applypulse(pulse, loc_=d['loc'], Δf_=d['df'], b1Map_=d['b1'])
        if self.keep_M:
            self.M = M
        loss = ((M - self.tgt) ** 2).sum()
        loss.backward()
        return loss

    def step(self, sp=None, pulse=None, d=None):
        sp, pulse, d = (self.sp, self.pulse, self.d) if sp is None else (sp, pulse, d)
        loss = self.local_step(sp, pulse, d).detach().reshape(1)
        if self.world > 1:
            self.parallel.allreduce_waveform_grads(pulse.rf, pulse.gr, loss)
        return loss


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


DUMP_MAX_SPINS = 1 << 20       # M rows written by --dump-outputs: 12 MB in fp32, 25 MB in fp64


def step_outputs(M, pulse, loss):
    """What one step hands its caller, as host arrays in the working dtype: M (the magnetisation applypulse returns; shape
    (N, nM, 3), or above DUMP_MAX_SPINS spins the rows of a fixed seeded sample of the flattened (N * nM, 3) spins, in
    ascending order), rf.grad, gr.grad and the loss."""
    M = M.detach()
    if M.shape[0] * M.shape[1] > DUMP_MAX_SPINS:
        M = M.reshape(-1, 3)
        idx = torch.randperm(M.shape[0], generator=torch.Generator().manual_seed(0))[:DUMP_MAX_SPINS].sort().values
        M = M[idx.to(M.device)]
    return {'M': M.cpu().numpy(), 'rf_grad': pulse.rf.grad.cpu().numpy(), 'gr_grad': pulse.gr.grad.cpu().numpy(),
            'loss': loss.detach().cpu().numpy()}


def timed_region(P, steps, flush, use_graph=True, out=None):
    """-> (ms summed over `steps` steps, our kernel launches, launch mode).  The whole step -- pack, forward, loss,
    adjoint backward, finalize and (N > 1) the in-place all-reduce -- is recorded once into a CUDA graph and replayed;
    if NCCL refuses the capture the all-reduce stays eager behind the replay; --no-graph times eager launches.
    `out` (a dict) receives host copies of what the last timed step returned to its caller (see step_outputs)."""
    from mrphy import _cabi
    pulse, world = P.pulse, P.world
    graph, per_step, mode, g_loss = None, None, 'eager', None
    P.keep_M = out is not None
    if use_graph:
        for with_comm, cmode in (((True, 'global'), (True, 'thread_local'), (False, 'global')) if world > 1 else ((False, 'global'),)):
            try:
                pulse.rf.grad = pulse.gr.grad = None
                l0 = _cabi.launch_counter
                g_ = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_, capture_error_mode=cmode):
                    g_loss = P.step() if with_comm else P.local_step().detach().reshape(1)
                per_step = _cabi.launch_counter - l0
                for _ in range(2):
                    g_.replay()
                    if world > 1 and not with_comm:
                        P.parallel.allreduce_waveform_grads(pulse.rf, pulse.gr, g_loss)
                torch.cuda.synchronize()
                graph = g_
                mode = ('CUDA graph replay of the step (pack, fwd, loss, bwd, finalize' +
                        (', in-place NCCL all-reduce of the flat gradient buffer)' if with_comm else ')') +
                        ('; all-reduce eager behind the replay' if world > 1 and not with_comm else ''))
                comm_in_graph = with_comm
                break
            except Exception as e:                  # noqa: BLE001 -- any capture problem: try the next mode
                print(f'[bench] CUDA graph capture failed ({type(e).__name__}: {str(e)[:200]})', file=sys.stderr)
                torch.cuda.synchronize()
                graph = None

    def one():
        if graph is None:
            pulse.rf.grad = pulse.gr.grad = None
            return P.step()
        graph.replay()
        if world > 1 and not comm_in_graph:
            P.parallel.allreduce_waveform_grads(pulse.rf, pulse.gr, g_loss)
        return g_loss

    barrier(world)
    l0 = _cabi.launch_counter
    evs, loss = [], None
    for _ in range(steps):
        flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = one()
        e1.record()
        evs.append((e0, e1))
    barrier(world)
    ms = sum(x.elapsed_time(y) for x, y in evs)
    n_launch = per_step * steps if graph is not None else _cabi.launch_counter - l0
    if out is not None:
        out.update(step_outputs(P.M, pulse, loss))
    P.keep_M, P.M = False, None
    loss = float(loss)
    pulse.rf.grad = pulse.gr.grad = None
    del graph
    return ms, n_launch, mode, loss


def e2e_region(P, steps, flush, pinned):
    """End to end: pinned host inputs -> device every step, loss + gradients read back into pinned host memory.  Two object
    sets: the copy stream uploads step i+1 while the compute stream runs step i; the timed region is the whole K-step
    loop, wall clock, synchronised on both sides.  -> (seconds for `steps` pipelined steps, serial seconds per step, h2d, d2h)"""
    host, dtype, world = P.host, P.dtype, P.world
    sets = [P.make_objects(host), P.make_objects(host)]
    outs = [(torch.empty(1, dtype=dtype).pin_memory(), torch.empty_like(host['rf']).pin_memory(),
             torch.empty_like(host['gr']).pin_memory()) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    free = [torch.cuda.Event(), torch.cuda.Event()]

    def upload(b, stream):
        sp_b, pulse_b, d_b = sets[b]
        with torch.cuda.stream(stream), torch.no_grad():
            for k in ('loc', 'df', 'b1'):
                d_b[k].copy_(pinned[k], non_blocking=True)
            sp_b.M_.copy_(pinned['M0'], non_blocking=True)
            pulse_b.rf.copy_(pinned['rf'], non_blocking=True)
            pulse_b.gr.copy_(pinned['gr'], non_blocking=True)

    def compute(b):
        sp_b, pulse_b, d_b = sets[b]
        pulse_b.rf.grad = pulse_b.gr.grad = None
        loss = P.step(sp_b, pulse_b, d_b)
        o = outs[b]
        o[0].copy_(loss, non_blocking=True)      # results: three async copies into pinned memory
        o[1].copy_(pulse_b.rf.grad, non_blocking=True)
        o[2].copy_(pulse_b.gr.grad, non_blocking=True)
        return o

    def serial():
        upload(0, torch.cuda.current_stream())
        o = compute(0)
        torch.cuda.current_stream().synchronize()
        return o

    def pipelined(K):
        cur = torch.cuda.current_stream()
        for ev in free:
            ev.record(cur)
        copy_stream.wait_stream(cur)
        upload(0, copy_stream)
        ready[0].record(copy_stream)
        o = None
        for i in range(K):
            b = i & 1
            if i + 1 < K:                       # next step's inputs, once the set they overwrite is no longer in use
                copy_stream.wait_event(free[b ^ 1])
                upload(b ^ 1, copy_stream)
                ready[b ^ 1].record(copy_stream)
            flush.fill_(1.0)                    # inside the timed region here (cannot be hidden in a pipeline)
            cur.wait_event(ready[b])
            o = compute(b)
            free[b].record(cur)
        torch.cuda.synchronize()
        return o

    serial()
    pipelined(2)
    barrier(world)
    t_serial = []
    for _ in range(min(steps, 3)):
        flush.fill_(1.0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        serial()
        t_serial.append(time.perf_counter() - t0)
    barrier(world)
    t0 = time.perf_counter()
    out = pipelined(steps)
    t_e2e = time.perf_counter() - t0
    barrier(world)
    h2d = sum(v.numel() * v.element_size() for v in pinned.values())
    d2h = sum(o.numel() * o.element_size() for o in out)
    return t_e2e, float(np.mean(t_serial)), h2d, d2h


def kernel_times(P, steps, flush):
    """per-kernel durations: CUDA events inside the C ABI, on the launching stream"""
    from mrphy import _cabi
    L = _cabi.lib()
    L.mrphy_kernel_timing(1)
    k_fwd, k_bwd = [], []
    for _ in range(steps):
        flush.fill_(1.0)
        P.pulse.rf.grad = P.pulse.gr.grad = None
        M = P.sp.applypulse(P.pulse, loc_=P.d['loc'], Δf_=P.d['df'], b1Map_=P.d['b1'])
        k_fwd.append(L.mrphy_last_kernel_ms())
        ((M - P.tgt) ** 2).sum().backward()
        k_bwd.append(L.mrphy_last_kernel_ms())
    L.mrphy_kernel_timing(0)
    del M          # a live autograd graph would pin AccumulateGrad nodes to this stream and spoil the next capture
    P.pulse.rf.grad = P.pulse.gr.grad = None
    return float(np.mean(k_fwd)), float(np.mean(k_bwd))


def parity_block(P, dtype):
    """The checker leg (oracle/ as the CHECKER only): a random 128-spin subset of THIS workload against the CPU oracle in
    fp64 and -- the reference algorithm's own fp32 floor -- in fp32, for the default policy and for 'strict'."""
    from mrphy import _ops
    from oracle import bloch_oracle as orc
    g, nS = P.host, 128          # this rank's slab (the whole cube at N = 1)
    gen = torch.Generator().manual_seed(7)
    nM = g['loc'].shape[1]
    sub = torch.randperm(nM, generator=gen)[:nS]
    w = torch.zeros(P.N, nM, 3, dtype=torch.float64)
    w[:, sub] = torch.rand(P.N, nS, 3, generator=gen, dtype=torch.float64) * 2 - 1
    bs = slice(0, 1)                                                    # first batch entry
    c32 = lambda v: float(np.float32(v)) if dtype == torch.float32 else v
    okw = dict(df=g['df'][bs][:, sub], b1=g['b1'][bs][:, sub], T1=c32(1.47), T2=c32(0.07), gamma=c32(4257.6), dt=c32(4e-6))
    oargs = (g['M0'][bs][:, sub], g['rf'][bs], g['gr'][bs], g['loc'][bs][:, sub], w[bs][:, sub])
    t0 = time.perf_counter()
    ref = orc.applypulse_fwd_bwd(*oargs, **okw)
    ref32 = orc.applypulse_fwd_bwd(*oargs, **okw, dtype=torch.float32) if dtype == torch.float32 else None
    mx = lambda a, b: float((a.detach().cpu().double() - b.double()).abs().max())
    rel = lambda a, b: float((a.detach().cpu().double() - b.double()).norm() / b.double().norm())
    out = {'subset': f'{nS} random spins of rank 0\'s slab of the workload, batch entry 0, oracle/bloch_oracle.py on CPU',
           'oracle_seconds': None, 'north_star': 'M 1e-5 abs (fp32) / 1e-12 (fp64); rf/gr gradients 1e-4 relative'}
    if ref32 is not None:
        out['reference_algorithm_fp32_vs_fp64'] = {'max_abs_dM': mx(ref32['Mo'], ref['Mo']), 'grf_rel': rel(ref32['grf'], ref['grf']),
                                                   'ggr_rel': rel(ref32['ggr'], ref['ggr'])}
    wd = w.to(device=P.dev, dtype=dtype)
    for pol in ((_ops.trig_policy(), 'strict') if dtype == torch.float32 else (None,)):
        _ops.set_trig_policy(pol)
        try:
            P.pulse.rf.grad = P.pulse.gr.grad = None
            M = P.sp.applypulse(P.pulse, loc_=P.d['loc'], Δf_=P.d['df'], b1Map_=P.d['b1'])
            (M * wd).sum().backward()
        finally:
            _ops.set_trig_policy(None)
        out['ours_' + (pol or 'fp64') + '_vs_reference_fp64'] = {
            'max_abs_dM': mx(M[bs][:, sub.to(P.dev)], ref['Mo']), 'grf_rel': rel(P.pulse.rf.grad[bs], ref['grf']),
            'ggr_rel': rel(P.pulse.gr.grad[bs], ref['ggr'])}
        del M
    P.pulse.rf.grad = P.pulse.gr.grad = None
    out['oracle_seconds'] = time.perf_counter() - t0
    return out


def multi_gpu_check(dtype, dev, rank, world):
    """Sharded-and-all-reduced gradients == single-GPU gradients: every rank runs its slab of a 32^3 x 256 cube cut by
    mrphy.parallel.shard_spins and all-reduces; rank 0 also runs the whole cube unsharded and compares."""
    P = Problem('small32', 'strong', dtype, dev, rank, world)
    P.pulse.rf.grad = P.pulse.gr.grad = None
    loss = P.step()
    torch.cuda.synchronize()
    if rank != 0:
        return None
    Q = Problem('small32', 'strong', dtype, dev, 0, 1)
    l1 = Q.step()
    rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
    return {'what': 'rf.grad / gr.grad / loss of a 32^3 x 256 cube: sharded over all ranks + one all-reduce vs unsharded on rank 0 '
                    '(relative L2; fp32 sums over spins in a different order)',
            'grf_rel': rel(P.pulse.rf.grad, Q.pulse.rf.grad), 'ggr_rel': rel(P.pulse.gr.grad, Q.pulse.gr.grad),
            'loss_rel': abs(float(loss) - float(l1)) / abs(float(l1)),
            'flat_buffer_allreduce': P.parallel.flat_wave_grads(P.pulse.rf, P.pulse.gr) is not None}


WORKLOADS['small32'] = (1, 32, 256)


def multicoil_leg(dev, flush, nC=8, n=64, nT=1000, reps=5):
    """Parallel transmit (b1Map with nC coils, SURVEY 8a3) at the C2 size, kernels only (CUDA events inside the C ABI around the
    forward -- transmit field on tcgen05 -- and the backward kernel), best of `reps` after one warm-up, L2 flushed."""
    from mrphy import _ops, _cabi
    g = torch.Generator(device=dev).manual_seed(0)
    U = lambda *s: torch.rand(s, generator=g, device=dev, dtype=torch.float32) * 2 - 1
    nM = n ** 3
    rf = (U(1, 2, nT, nC) * 0.1 / nC).requires_grad_(True)
    gr = (U(1, 3, nT) * 2).requires_grad_(True)
    b1, loc, df = U(1, nM, 2, nC), U(1, nM, 3) * 12, U(1, nM) * 200
    M0 = torch.tensor([0., 0., 1.], device=dev).expand(1, nM, 3).contiguous()
    c = lambda v: torch.tensor(v, device=dev)
    L = _cabi.lib()
    L.mrphy_kernel_timing(1)
    f, b = [], []
    try:
        for i in range(reps + 1):
            flush.fill_(1.0)
            rf.grad = gr.grad = None
            Mo = _ops.fused_applypulse(M0, rf, gr, loc, Δf_=df, b1Map_=b1, T1_=c(1.47), T2_=c(0.07), γ_=c(4257.6), dt=c(4e-6))
            tf = L.mrphy_last_kernel_ms()
            Mo.sum().backward()
            tb = L.mrphy_last_kernel_ms()
            if i:
                f.append(tf)
                b.append(tb)
    finally:
        L.mrphy_kernel_timing(0)
    return {'workload': f'{n}^3 spins x {nT} steps, {nC} transmit coils with a b1Map, fp32', 'value': nM * nT / ((min(f) + min(b)) * 1e-3),
            'unit': UNIT, 'fwd_kernel_ms': min(f), 'bwd_kernel_ms': min(b),
            'how': 'kernels only; forward: transmit field as a split-operand TF32 tcgen05.mma product (fused_fwd_tc_kernel)'}


def measure(workload, scaling, args, dev, rank, world, flush, full):
    """Timed region (+ with `full`: e2e, per-kernel times, alternative policies, parity) of one workload."""
    import torch.distributed as dist
    from mrphy import _ops
    dtype = torch.float32 if args.dtype == 'f32' else torch.float64
    P = Problem(workload, scaling, dtype, dev, rank, world)
    for _ in range(args.warmup):
        P.pulse.rf.grad = P.pulse.gr.grad = None
        P.step()
    barrier(world)
    outputs = {} if full and args.dump_outputs and rank == 0 else None
    ms_total, launches, mode, loss = timed_region(P, args.steps, flush, not args.no_graph, outputs)
    res = {'ms_total': ms_total, 'launches': launches, 'mode': mode, 'loss': loss, 'nM': P.nM, 'N': P.N, 'nT': P.nT,
           'policy': _ops.trig_policy() if dtype == torch.float32 else 'fp64', 'outputs': outputs}
    if full:
        pinned = {k: v.pin_memory() for k, v in P.host.items()}
        res['e2e'] = e2e_region(P, args.steps, flush, pinned)
        del pinned
        res['k_fwd'], res['k_bwd'] = kernel_times(P, min(args.steps, 10), flush)
        res['alt'] = {}
        if dtype == torch.float32:
            for pol in ('precise', 'mixed', 'fast', 'strict'):
                if pol == _ops.trig_policy():
                    continue
                _ops.set_trig_policy(pol)
                try:
                    for _ in range(2):
                        P.pulse.rf.grad = P.pulse.gr.grad = None
                        P.step()
                    k = min(args.steps, 5) if pol == 'strict' else args.steps
                    res['alt'][pol] = timed_region(P, k, flush, not args.no_graph)[0] / k
                finally:
                    _ops.set_trig_policy(None)
        res['parity'] = parity_block(P, dtype) if rank == 0 else None
    t = torch.tensor([res['ms_total']] + ([res['e2e'][0] * 1e3] + [res['alt'].get(p, 0.0) for p in ('precise', 'mixed', 'fast', 'strict')]
                                           if full else []), dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    res['ms_total'] = float(t[0])
    if full:
        res['ms_e2e'] = float(t[1])
        res['alt'] = {p: float(t[2 + i]) for i, p in enumerate(('precise', 'mixed', 'fast', 'strict')) if float(t[2 + i]) > 0}
    res['units'] = P.units_local * world if scaling == 'weak' else float(P.N) * (P.n ** 3) * P.nT
    res['units_local'] = P.units_local
    res['esz'] = 4 if dtype == torch.float32 else 8
    # checkpoint interval the kernels ran with: T1 / T2 of the synthetic spins allow the cap of the kernel family
    res['K'] = _ops.K_MAX1 if dtype == torch.float32 and _ops.trig_policy() != 'strict' else _ops.K_MAX
    del P
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    use_ours()
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        # rank 0 prints ONE JSON line on stdout: NCCL's version banner / debug output goes to stderr instead
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        if os.environ.get('NCCL_DEBUG', '').upper() in ('VERSION', 'WARN'):
            del os.environ['NCCL_DEBUG']          # the banner ignores NCCL_DEBUG_FILE (checked: profiles/nccl_stdout_check.py)
        dist.init_process_group('nccl', device_id=dev)
        dist.all_reduce(torch.zeros(1, device=dev))            # communicator up before any capture
    scaling = pick_scaling(args)
    dtype = torch.float32 if args.dtype == 'f32' else torch.float64
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 256 MB > 126 MB L2
    sampler = ClockSampler(local)      # samples through warm-up, the timed region and the e2e / per-kernel legs
    if rank == 0:
        sampler.start()
    r = measure(args.workload, scaling, args, dev, rank, world, flush, full=True)
    clocks = sampler.stop() if rank == 0 else None
    if r['outputs'] is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in r['outputs'].items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a)
    c2 = None
    if args.workload != 'c2' and world == 1 and not args.no_extras:     # the 1-GPU configuration of BASELINE.json, same run
        c2 = measure('c2', 'weak', args, dev, rank, world, flush, full=False)
    check = multi_gpu_check(dtype, dev, rank, world) if world > 1 else None
    if rank == 0:
        props = torch.cuda.get_device_properties(dev)
        sms = props.multi_processor_count
        hbm_gbs, sm_mhz, src = peaks()
        issue_roof = sms * 128 * sm_mhz * 1e6 / ISSUE_SLOTS           # spin-steps/s per GPU
        peak_tf = sms * 128 * 2 * sm_mhz * 1e6 / 1e12
        value = r['units'] * args.steps / (r['ms_total'] * 1e-3)
        e2e = r['units'] * args.steps / (r['ms_e2e'] * 1e-3)
        ms_f, ms_b = r['k_fwd'], r['k_bwd']
        per_launch = r['units_local']
        ach_tf = per_launch * FLOP_BWD / (ms_b * 1e-3) / 1e12
        ck_bytes = per_launch / r['K'] * 3 * r['esz'] + r['N'] * r['nM'] * (3 + 3 + 3 + 2 + 1 + 3) * r['esz']   # bwd: ckpt reads + operands
        traffic, traffic_src = None, None
        try:   # dram__bytes_read+write per launch of the same kernel from the committed ncu capture of the same workload
            with open(os.path.join(ROOT, 'profiles', 'r2_ncu_summary.json')) as f:
                cap = json.load(f)['captures'].get(f'{args.workload}_{args.dtype}_bwd')
            if cap:
                m = cap['metrics']
                scale = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
                traffic = sum(m[k]['value'] * scale[m[k]['unit']] for k in ('dram__bytes_read.sum', 'dram__bytes_write.sum'))
                traffic_src = 'static: profiles/r2_ncu_summary.json (ncu --set full capture of this kernel on this workload), not measured in this run'
        except Exception:
            pass
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': r['ms_total'] / args.steps, 'higher_is_better': True,
            'scaling': scaling, 'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
            'config': {'workload': workload_desc(args.workload, scaling, world), 'spins_per_gpu': r['N'] * r['nM'], 'nT': r['nT'],
                       'l2': 'flushed between steps (256 MB write)', 'launch': r['mode'],
                       'sharding': (f'contiguous compact-spin slabs x{world} (mrphy.parallel.shard_spins), waveform replicated, ONE '
                                    'in-place all-reduce of the flat [rf.grad|gr.grad|loss] buffer') if world > 1 else 'single GPU',
                       'trig': (r['policy'] + ' (default)') if args.dtype == 'f32' else 'fp64'},
            'e2e': {'value': e2e, 'unit': UNIT, 'h2d_bytes_per_step': r['e2e'][2], 'd2h_bytes_per_step': r['e2e'][3],
                    'how': 'K steps back to back, wall clock: uploads of step i+1 (copy stream) overlap step i, L2 flush and '
                           'read-back inside the timed region', 'serial_ms_per_step': r['e2e'][1] * 1e3},
            'gpu_launches': r['launches'],
            'loss': r['loss'],
            'clocks': clocks,
            'roofline': {'bound': 'fp32_issue', 'kernel': 'fused_bwd_kernel', 'achieved': ach_tf, 'peak': peak_tf,
                         'unit': 'TFLOP/s', 'frac': ach_tf / peak_tf, 'traffic': traffic, 'traffic_unit': 'bytes/launch',
                         'traffic_source': traffic_src, 'algorithmic_bytes_per_launch': ck_bytes, 'checkpoint_interval': r['K'],
                         'peak_source': f'{sms} SMs (device query) x 128 FP32 lanes x 2 x sm_max_mhz ({src} {sm_mhz:.0f} MHz); the path '
                                        'is FP32-issue-bound (SURVEY 8d), not HBM- or tensor-bound',
                         'ms_per_launch': ms_b, 'algorithmic_flop_per_spin_step': FLOP_BWD,
                         'fwd_kernel': {'ms_per_launch': ms_f, 'achieved': per_launch * FLOP_FWD / (ms_f * 1e-3) / 1e12,
                                        'frac': per_launch * FLOP_FWD / (ms_f * 1e-3) / 1e12 / peak_tf},
                         'issue_roofline_spin_steps_per_gpu': issue_roof,
                         'fwd_bwd_frac_of_issue_roofline': value / world / issue_roof,
                         'kernels_only_frac_of_issue_roofline': per_launch / ((ms_f + ms_b) * 1e-3) / issue_roof,
                         'hbm': {'achieved_gbs': ck_bytes / (ms_b * 1e-3) / 1e9, 'peak_gbs': hbm_gbs,
                                 'frac': ck_bytes / (ms_b * 1e-3) / 1e9 / hbm_gbs, 'source': src}},
            'policies': {p: {'value': r['units'] / (ms * 1e-3), 'ms_per_step': ms, 'frac_of_issue_roofline': r['units'] / (ms * 1e-3) / world / issue_roof}
                         for p, ms in r['alt'].items()},
            'parity': r['parity'],
        }
        if c2 is not None:
            v2 = c2['units'] * args.steps / (c2['ms_total'] * 1e-3)
            line['c2'] = {'workload': workload_desc('c2', 'weak', 1), 'value': v2, 'ms_per_step': c2['ms_total'] / args.steps,
                          'frac_of_issue_roofline': v2 / issue_roof, 'policy': c2['policy'], 'loss': c2['loss']}
        if check is not None:
            line['multi_gpu_check'] = check
        if world == 1 and not args.no_extras and args.dtype == 'f32':
            line['ptx_8_coils'] = multicoil_leg(dev, flush)
        if world == 1 and not args.no_extras:      # CPU / eager baselines are timed at N=1 only; the other ranks must not wait on them
            line['cpu_baseline'] = reference_subprocess(args, 'cpu')
            line['torch_eager_same_gpu'] = reference_subprocess(args, 'cuda')
        else:
            line['cpu_baseline'] = None
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def reference_subprocess(args, device):
    """The reference arm as a child process (the reference package is also called `mrphy`: it cannot share this process)."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--workload', args.workload, '--dtype', args.dtype,
           '--steps', '1', '--warmup', '0' if device == 'cpu' else '1', '--ref-device', device]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env={k: v for k, v in os.environ.items()
                             if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')})
        j = json.loads(out.stdout.strip().splitlines()[-1])
        cb = j['cpu_baseline']
        if device == 'cuda':
            return {'value': j['value'], 'unit': UNIT, 'kind': cb['kind'] + ' in torch-eager CUDA on this GPU (context only)',
                    'sample': cb['sample']}
        return cb
    except Exception as e:      # context only
        return {'error': f'{type(e).__name__}: {str(e)[:200]}'}


# ======================================================================================================================
# reference arm: the unmodified reference's own public API (oracle/_ref), else the oracle port
def reference_step(kind, n, nT, dtype, device, N=1, interp=1):
    """One fwd+bwd of `SpinCube.applypulse` on an n^3 sub-cube with the bench distributions -> (seconds, spin-steps)."""
    tgt = torch.tensor([0., 1., 0.], dtype=dtype, device=device)
    if kind == 'reference':
        from mrphy import mobjs        # oracle/_ref/mrphy: the unmodified reference
        s = synth(N, n, n, nT, dtype, interp=interp, mobjs=mobjs)
        kw = {'dtype': dtype, 'device': torch.device(device)}
        cube = mobjs.SpinCube((N, n, n, n), torch.tensor([[24., 24., 24.]]), Δf_=s['df'].to(device), **kw)
        pulse = mobjs.Pulse(rf=s['rf'].to(device).requires_grad_(True), gr=s['gr'].to(device).requires_grad_(True),
                            dt=torch.tensor(4e-6), **kw)
        b1 = s['b1'].to(device)
        sync = torch.cuda.synchronize if device == 'cuda' else (lambda: None)
        sync()
        t0 = time.perf_counter()
        M_ = cube.applypulse(pulse, b1Map_=b1)          # mobjs.py:841-869 -> sims.py:24-269
        loss = ((M_ - tgt) ** 2).sum()
        loss.backward()
        sync()
        return time.perf_counter() - t0, N * n ** 3 * nT
    from oracle import bloch_oracle as orc
    s = synth(N, n, n, nT, dtype)
    orc.DEVICE = device
    try:
        s = {k: v.to(device) for k, v in s.items()}
        sync = torch.cuda.synchronize if device == 'cuda' else (lambda: None)
        sync()
        t0 = time.perf_counter()
        orc.applypulse_fwd_bwd(s['M0'], s['rf'], s['gr'], s['loc'], lambda Mo: 2 * (Mo - tgt), df=s['df'], b1=s['b1'],
                               T1=1.47, T2=0.07, dtype=dtype)
        sync()
        return time.perf_counter() - t0, N * n ** 3 * nT
    finally:
        orc.DEVICE = 'cpu'


def run_reference(args):
    """The reference's own implementation of the path on the host cores (or, --ref-device cuda, in torch-eager CUDA)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    kind = use_reference()
    N, n, nT = WORKLOADS[args.workload]
    dtype = torch.float32 if args.dtype == 'f32' else torch.float64
    cores = len(os.sched_getaffinity(0))
    torch.set_num_threads(cores)
    device = args.ref_device
    scaling = pick_scaling(args)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    # bounded sample: an n_s^3 sub-cube (same distributions, same nT, same dtype), sized for ~15 s of CPU work per step
    # at the reference's ~5e5 spin-steps/s on 8 cores (BASELINE.md sec. 2), and for the whole run to end in minutes; the
    # reference stores 52 B per spin-step (sims.py:63,84-88), so the full cubes do not fit anyway
    budget = min(15.0, 150.0 / max(args.steps + args.warmup, 1))
    rate = 6e4 * cores if device == 'cpu' else 5e7
    n_s = min(n, int(max(8, min(48 if device == 'cuda' else 32, round((budget * rate / nT / max(N, 1)) ** (1 / 3))))))
    N_s = min(N, 4)
    itp = 5 if args.workload == 'c3' else 1
    for _ in range(args.warmup):
        reference_step(kind, n_s, nT, dtype, device, N_s, itp)
    tot, units = 0.0, 0
    for _ in range(args.steps):
        s, u = reference_step(kind, n_s, nT, dtype, device, N_s, itp)
        tot += s
        units += u
    v = units / tot
    what = ('the UNMODIFIED reference (oracle/_ref/mrphy: SpinCube.applypulse + loss.backward through its own public API)'
            if kind == 'reference' else 'oracle/bloch_oracle.py (port of the reference algorithm; no staged reference found)')
    sample = (f'{what}, torch {device} ' + (f'{cores} threads' if device == 'cpu' else 'eager') +
              f', {N_s} x {n_s}^3 sub-cube of the workload (same distributions, dtype {args.dtype}, same nT={nT}) per step, '
              f'{tot / max(args.steps, 1):.1f} s per step')
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': tot / max(args.steps, 1) * 1e3, 'higher_is_better': True,
        'scaling': scaling, 'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
        'config': {'workload': workload_desc(args.workload, scaling, world), 'nT': nT,
                   'sample': f'each step = one fwd+bwd over a {N_s} x {n_s}^3 sub-cube of the workload; the full cube needs 52 B per '
                             'spin-step in the reference (C5: 3.5 TB)'},
        'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': cores, 'kind': kind, 'sample': sample},
        'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }), flush=True)


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='c5', choices=sorted(w for w in WORKLOADS if w != 'small32'))
    ap.add_argument('--dtype', default='f32', choices=['f32', 'f64'])
    ap.add_argument('--scaling', default=None, choices=['weak', 'strong'],
                    help='default: strong for c5 (the north_star scaling problem), weak otherwise')
    ap.add_argument('--no-graph', action='store_true', help='time eager launches instead of a CUDA graph replay')
    ap.add_argument('--no-extras', action='store_true', help='skip the C2 leg and the CPU / eager reference legs')
    ap.add_argument('--ref-device', default='cpu', choices=['cpu', 'cuda'], help='(reference arm) where the reference runs')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned (M, rf_grad, gr_grad, loss; rank 0) as DIR/<name>.npy; '
                         f'M of more than {DUMP_MAX_SPINS} spins is a fixed seeded sample of them')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    a.warmup = max(a.warmup, 3) if a.impl == 'ours' else a.warmup
    (run_ours if a.impl == 'ours' else run_reference)(a)
