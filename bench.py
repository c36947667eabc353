#!/usr/bin/env python
"""Benchmark of the VB-HMM EM hot path (BASELINE.json metric: x-vectors/s through 10 EM iterations).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one JSON line on rank 0)
    python bench.py --impl reference ...                     # the reference's CPU implementation on the host cores

A step = one pass of the hot path over one synthetic batch: rho = X.V (projection) followed by the workload's EM
iterations (epsilon = -inf: the reference then never breaks, VBx/VBx.py:122).  `value` is measured with X / gamma0
resident in HBM; `e2e` goes through the host-buffer API (pinned host X and gamma0 copied in, gamma/pi/Li copied out,
inside the timed region).  Multi-GPU: recordings are independent; the headline workload gives every rank its own
batch (weak scaling), `--workload c4` shards ONE fixed batch of 192 long recordings over the ranks (strong scaling);
either way the only collective is one NCCL all-reduce of the ELBO trace, issued inside the library (vbx_elbo_trace).
`--workload c1` times the reference's own call (VBx/vbhmm.py:154-158 on ES2005a) through the drop-in VBx().
"""
import os
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")   # before numpy: the CPU baseline runs one process per core
os.environ.setdefault("OMP_NUM_THREADS", "1")
import argparse
import contextlib
import json
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'x-vectors/sec through 10 VB-HMM EM iters'
UNIT = 'x-vectors/s'

# SURVEY.md 8(d) / BASELINE.json configs.  B = recordings per GPU, except for strong-scaling workloads (B = the whole job)
WORKLOADS = {
    # north_star headline: 4096 recordings x T=1000, D=256 / R=128 / S=16, 10 iterations, one GPU
    'headline': dict(B=4096, T=1000, S=16, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'c1': dict(B=1, T=1025, S=31, iters=40, Fa=0.3, Fb=17.0, loopP=0.99, dropin=True),    # ES2005a, the reference's own call
    'c2': dict(B=256, T=1000, S=16, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'c3': dict(B=4096, T=(200, 3000), S=16, iters=20, Fa=0.3, Fb=17.0, loopP=0.99),
    # DIHARD-II-shaped: ONE batch of 192 long recordings sharded over the GPUs of the box (strong scaling)
    'c4': dict(B=192, T=12000, S=30, iters=40, Fa=0.2, Fb=6.0, loopP=0.35, strong=True),
    'c4share': dict(B=24, T=12000, S=30, iters=40, Fa=0.2, Fb=6.0, loopP=0.35),     # one GPU's share of c4 at 8 GPUs
    'c5s4': dict(B=1024, T=2000, S=4, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'c5s8': dict(B=1024, T=2000, S=8, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'c5s16': dict(B=1024, T=2000, S=16, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'c5s32': dict(B=1024, T=2000, S=32, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'c5s64': dict(B=1024, T=2000, S=64, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'tiny': dict(B=32, T=300, S=16, iters=10, Fa=0.3, Fb=17.0, loopP=0.99),
    'tinystrong': dict(B=12, T=(300, 5000), S=6, iters=6, Fa=0.3, Fb=17.0, loopP=0.99, strong=True),
}
D_RAW, R_DIM = 256, 128


def workload_lengths(w, seed):
    if isinstance(w['T'], tuple):
        rng = np.random.default_rng(seed)
        return rng.integers(w['T'][0], w['T'][1] + 1, size=w['B']).astype(np.int64)
    return np.full(w['B'], w['T'], dtype=np.int64)


# ------------------------------------------------------------------------------------------------
# synthetic data on the device (same generative model as vbx_b200/synth.py, vectorised in torch)
# ------------------------------------------------------------------------------------------------
def make_device_batch(lengths, S, seed, device):
    import torch
    from vbx_b200 import synth
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    B, Tm = len(lengths), int(max(lengths))
    Phi = torch.from_numpy(synth.plda_phi(R_DIM)).to(device=device, dtype=torch.float32)
    V0 = torch.from_numpy(synth.projection_basis(D_RAW, R_DIM)).to(device=device, dtype=torch.float32)
    lens_d = torch.from_numpy(np.asarray(lengths)).to(device)
    keep = (torch.arange(Tm, device=device)[None, :] < lens_d[:, None]).reshape(-1)
    ragged = not bool(keep.all())
    n_spk = torch.randint(2, 9, (B,), device=device, generator=g)
    means = torch.randn((B, 8, R_DIM), device=device, generator=g) * Phi.sqrt()
    X_parts, G_parts = [], []
    chunk = max(1, (1 << 22) // Tm)            # recordings per chunk, bounds temporaries to ~1 GB
    for b0 in range(0, B, chunk):
        b1 = min(B, b0 + chunk)
        nb = b1 - b0
        switch = torch.rand((nb, Tm), device=device, generator=g) >= 0.99
        switch[:, 0] = True
        jump = (torch.rand((nb, Tm), device=device, generator=g) * n_spk[b0:b1, None]).long()
        idx = torch.where(switch, torch.arange(Tm, device=device)[None, :].expand(nb, Tm), torch.zeros((), dtype=torch.long, device=device))
        last = torch.cummax(idx, dim=1).values
        z = torch.gather(jump, 1, last)                                        # sticky Markov path
        fea = torch.gather(means[b0:b1], 1, z[:, :, None].expand(nb, Tm, R_DIM))
        fea = fea + torch.randn((nb, Tm, R_DIM), device=device, generator=g)
        noise = torch.randn((nb * Tm, D_RAW), device=device, generator=g)
        noise = noise - (noise @ V0) @ V0.T
        X = fea.reshape(-1, R_DIM) @ V0.T + 0.5 * noise
        gam = -torch.log(torch.rand((nb * Tm, S), device=device, generator=g).clamp_min(1e-12))
        gam = gam / gam.sum(1, keepdim=True)                                  # flat Dirichlet rows, VBx/VBx.py:82-83
        if ragged:
            k = keep[b0 * Tm:b1 * Tm]
            X, gam = X[k], gam[k]
        X_parts.append(X)
        G_parts.append(gam)
        del fea, noise, z, jump, switch, idx, last
    X = torch.cat(X_parts) if len(X_parts) > 1 else X_parts[0]
    gamma0 = torch.cat(G_parts) if len(G_parts) > 1 else G_parts[0]
    V = (V0 * Phi.sqrt()[None, :]).contiguous()
    return dict(X=X.contiguous(), V=V, V0=V0, Phi=Phi, gamma0=gamma0.contiguous())


def make_device_shard(all_lengths, indices, S, seed, device):
    """Strong scaling: recording i of the job is generated from seed + i whichever rank owns it."""
    import torch
    parts = [make_device_batch(all_lengths[i:i + 1], S, seed + 7919 * int(i), device) for i in indices]
    out = dict(parts[0])
    out['X'] = torch.cat([p['X'] for p in parts]).contiguous()
    out['gamma0'] = torch.cat([p['gamma0'] for p in parts]).contiguous()
    return out


# ------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md "clocks line")
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                clk, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            smax = mx
            if t0 - 0.05 <= ts <= t1 + 0.05:
                sm.append(clk)
                for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                    if val.lower().startswith('active'):
                        reasons.add(name)
        if not sm:   # region shorter than the sampling period: use every sample we have
            sm = [float(l.split(',')[1]) for _, l in self.lines if len(l.split(',')) >= 9]
        if not sm:   # the sampling stream produced nothing: one direct query right after the region
            try:
                q = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i', str(self.index)],
                                   capture_output=True, text=True, timeout=20).stdout.strip().split(',')
                sm, smax = [float(q[1])], float(q[2])
                for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), q[5:9]):
                    if val.strip().lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                sm = [float('nan')]
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': smax, 'reasons': sorted(reasons), 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------
# NUMA: the host thread that feeds a GPU, and the pinned buffers it allocates, belong on the GPU's own NUMA node
# ------------------------------------------------------------------------------------------------
def gpu_numa_cpus(index):
    """(node, cpu list) of the NUMA node GPU `index` hangs off, or None."""
    try:
        bus = subprocess.run(['nvidia-smi', '--query-gpu=pci.bus_id', '--format=csv,noheader', '-i', str(index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith('00000000:'):
            bus = bus[4:]
        node = int(open(f'/sys/bus/pci/devices/{bus}/numa_node').read().strip())
        if node < 0:
            return None
        cpus = []
        for part in open(f'/sys/devices/system/node/node{node}/cpulist').read().strip().split(','):
            lo, _, hi = part.partition('-')
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        return (node, cpus) if cpus else None
    except Exception:
        return None


@contextlib.contextmanager
def numa_affinity(index, info):
    """Run the body (pinned allocations + the host side of the e2e pipeline) on the GPU's NUMA node."""
    try:
        old = os.sched_getaffinity(0)
    except Exception:
        old = None
    loc = gpu_numa_cpus(index) if old is not None else None
    if loc:
        try:
            os.sched_setaffinity(0, loc[1])
            info.update(node=loc[0], cpus=len(loc[1]))
        except Exception:
            loc = None
    try:
        yield
    finally:
        if loc and old is not None:
            try:
                os.sched_setaffinity(0, old)
            except Exception:
                pass


# ------------------------------------------------------------------------------------------------
# CPU arm.  The UNMODIFIED reference VBx.VBx when a copy is reachable ($VBX_REF, baseline/_ref installed with pip from
# /root/reference, /root/reference itself), else the oracle port; one recording per process on all host cores (the
# reference's own one-process-per-recording model, AMI_run.sh:53-58).
# ------------------------------------------------------------------------------------------------
def reference_dir():
    cands = []
    if os.environ.get('VBX_REF'):
        cands += [os.path.join(os.environ['VBX_REF'], 'VBx'), os.environ['VBX_REF']]
    cands += [os.path.join(ROOT, 'baseline', '_ref', 'VBx'), '/root/reference/VBx']
    for c in cands:
        if os.path.isfile(os.path.join(c, 'VBx.py')):
            return c
    return None


_REF_FN = None


def cpu_vbx():
    """-> (callable with the reference's VBx() signature, kind, description)."""
    global _REF_FN
    if _REF_FN is None:
        d = reference_dir()
        if d is not None:
            import importlib.util
            spec = importlib.util.spec_from_file_location('vbx_reference_module', os.path.join(d, 'VBx.py'))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            _REF_FN = (mod.VBx, 'reference', f'unmodified reference VBx.VBx ({d}/VBx.py), float64 numpy')
        else:
            from oracle import vbx_oracle as po
            _REF_FN = (po.vbx_oracle, 'port', 'oracle/vbx_oracle.py: float64 numpy restatement of VBx/VBx.py (log-domain '
                       'recursions, same per-frame Python overhead as the reference)')
    return _REF_FN


def _cpu_task(args):
    os.environ['OPENBLAS_NUM_THREADS'] = '1'
    X, V0, Phi, g0, S, iters, Fa, Fb, loopP, eps = args
    fn = cpu_vbx()[0]
    fea = X.astype(np.float64) @ V0.astype(np.float64) if V0 is not None else X.astype(np.float64)   # VBx/vbhmm.py:153
    t = time.perf_counter()
    fn(fea, Phi.astype(np.float64), loopProb=loopP, Fa=Fa, Fb=Fb, pi=S, gamma=g0.astype(np.float64), maxIters=iters, epsilon=eps)
    return time.perf_counter() - t


def _cpu_warm(_):
    os.environ['OPENBLAS_NUM_THREADS'] = '1'
    cpu_vbx()
    return 0


def cpu_pool_run(tasks, cores, repeats=1, warmup=0):
    import multiprocessing as mp
    ctx = mp.get_context('fork')
    used = min(cores, len(tasks))
    walls = []
    with ctx.Pool(used) as pool:
        pool.map(_cpu_warm, range(used))
        for i in range(warmup + repeats):
            t0 = time.perf_counter()
            pool.map(_cpu_task, tasks, chunksize=1)
            if i >= warmup:
                walls.append(time.perf_counter() - t0)
    return walls, used


def bounded(w, max_T=3000, max_iters=10):
    """The CPU arm's bounded sample: the reference's cost is linear in frames and in iterations, so long recordings are
    cut to max_T frames and long runs to max_iters iterations; throughput is scaled back to the workload's iteration
    count (x-vectors/s through w['iters'] iterations = x-vectors/s through k iterations * k / w['iters'])."""
    T = w['T']
    T2 = (min(T[0], max_T), min(T[1], max_T)) if isinstance(T, tuple) else min(T, max_T)
    it2 = min(w['iters'], max_iters)
    ws = dict(w, T=T2, iters=it2)
    note = ''
    if T2 != T or it2 != w['iters']:
        note = (f' [bounded: recordings cut to T<={max_T}, {it2} of {w["iters"]} iterations timed, throughput scaled by {it2}/{w["iters"]} '
                'to the workload\'s iteration count]')
    return ws, it2 / w['iters'], note


def host_sample(w, n_rec, seed):
    """A bounded sample of the workload generated on the host with the numpy generator (same model)."""
    from vbx_b200 import synth
    lens = workload_lengths(w, seed)[:n_rec]
    d = synth.make_batch(lens, R=R_DIM, S=w['S'], seed=seed, D=D_RAW, dtype=np.float32)
    recs = [(d['X'][lo:hi], d['gamma0'][lo:hi]) for lo, hi in zip(d['offsets'][:-1], d['offsets'][1:])]
    return recs, synth.projection_basis(D_RAW, R_DIM), d['Phi']


def es2005a_call():
    """Inputs of the reference's own VBx() call on ES2005a (VBx/vbhmm.py:150-158, run_example.sh:23-34), from the
    reference-generated fixture tests/golden/es2005a.npz."""
    z = np.load(os.path.join(ROOT, 'tests', 'golden', 'es2005a.npz'))
    lab = z['labels_ahc'].astype(int)
    q = np.zeros((len(lab), lab.max() + 1))
    q[np.arange(len(lab)), lab] = 1.0
    q = np.exp(q * float(z['smoothing']))
    q /= q.sum(1, keepdims=True)
    kw = dict(loopProb=float(z['loopProb']), Fa=float(z['Fa']), Fb=float(z['Fb']), maxIters=40, epsilon=1e-6)
    return z, z['fea'], z['Phi'], q, kw


def dist_env():
    return int(os.environ.get('RANK', 0)), int(os.environ.get('LOCAL_RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))


def workload_config(w, wname, n_gpus):
    T = w['T']
    per = 'recordings in the job' if w.get('strong') else 'recordings/GPU'
    cfg = {'workload': f'{wname}: B={w["B"]} {per} x T={"U[%d,%d]" % T if isinstance(T, tuple) else T} '
                       f'x D={D_RAW} -> R={R_DIM}, S={w["S"]}, {w["iters"]} EM iterations',
           'recordings': w['B'], 'recordings_are': 'whole job (sharded over the GPUs)' if w.get('strong') else 'per GPU',
           'frames_per_recording': list(T) if isinstance(T, tuple) else T, 'D': D_RAW,
           'R': R_DIM, 'S': w['S'], 'em_iterations': w['iters'], 'Fa': w['Fa'], 'Fb': w['Fb'], 'loopProb': w['loopP'],
           'parallelism': f'recordings sharded over {n_gpus} GPU(s), one NCCL all-reduce of the ELBO trace',
           'l2': 'inputs larger than L2 (rho alone exceeds 126 MB)' if w['B'] * (np.mean(T) if isinstance(T, tuple) else T) * R_DIM * 4 / (n_gpus if w.get('strong') else 1) > 2 * 126e6
                 else 'L2 flushed between steps (256 MB scratch write)'}
    if w.get('dropin'):
        cfg['workload'] = (f'{wname}: ES2005a (T=1025 x-vectors, R=128, S=31 AHC clusters), the reference call VBx/vbhmm.py:154-158 '
                           '(maxIters=40, epsilon=1e-6 -> 13 iterations), host numpy in / out')
        cfg['parallelism'] = 'one recording, one GPU'
        cfg['l2'] = 'single recording (0.5 MB): L2 resident by nature, as in the reference use'
    return cfg


# ------------------------------------------------------------------------------------------------
# --impl reference
# ------------------------------------------------------------------------------------------------
def run_reference(args, w, wname):
    """The reference's CPU implementation of the path on all host cores; each step = a bounded sample of the workload."""
    rank, _, world = dist_env()
    if rank != 0:
        return
    fn, kind, desc = cpu_vbx()
    cores = os.cpu_count() or 1
    if w.get('dropin'):
        z, fea, Phi, q, kw = es2005a_call()
        tasks = [(fea, None, Phi, q, q.shape[1], kw['maxIters'], kw['Fa'], kw['Fb'], kw['loopProb'], kw['epsilon'])]
        sample = 'the recording itself (ES2005a, 13 iterations until the epsilon stop), one process'
    else:
        n_rec = max(8, cores)
        ws, scale, bnote = bounded(w)
        recs, V0, Phi = host_sample(ws, n_rec, seed=1)
        tasks = [(X, V0, Phi, g0, ws['S'], ws['iters'], ws['Fa'], ws['Fb'], ws['loopP'], -np.inf) for X, g0 in recs]
        sample = f'{len(tasks)} recordings x {ws["iters"]} iterations of the workload per step, one per process{bnote}'
    frames = sum(t[0].shape[0] for t in tasks)
    walls, used = cpu_pool_run(tasks, cores, repeats=args.steps, warmup=args.warmup)
    ms = 1e3 * float(np.mean(walls))
    value = frames / (ms / 1e3) * (1.0 if w.get('dropin') else scale)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong' if w.get('strong') else 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'real (ES2005a fixture)' if w.get('dropin') else 'synthetic',
        'config': workload_config(w, wname, args.gpus),
        'note': f'bounded sample: {len(tasks)} recording(s) ({frames} x-vectors) per step',
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': used, 'kind': kind, 'sample': f'{sample}; {desc}, OPENBLAS_NUM_THREADS=1'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# --workload c1: the drop-in VBx() on the reference's own call
# ------------------------------------------------------------------------------------------------
def run_c1(args, w, wname):
    import torch
    import vbx_b200.api as api
    from vbx_b200.batch import VbxBatch
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    z, fea, Phi, q, kw = es2005a_call()
    T, S = q.shape
    call = lambda: api.VBx(fea, Phi, pi=S, gamma=q, **kw)
    default = api.PRECISION                  # what a caller of the drop-in gets without configuring anything
    modes = {}
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_all0 = time.time()
    for prec in ('float64', 'float32'):
        api.set_precision(prec)
        api.clear_plan_cache()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g, p, L = call()                      # cold: handle + plan + workspace are created inside
        cold = time.perf_counter() - t0
        for _ in range(max(args.warmup, 3)):
            call()
        ts = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            g, p, L = call()
            ts.append(time.perf_counter() - t0)
        modes[prec] = dict(cold_ms=1e3 * cold, warm_ms=1e3 * float(np.median(ts)), warm_ms_min=1e3 * float(np.min(ts)), iterations=len(L),
                           max_abs_gamma_vs_reference=float(np.abs(g - z['gamma']).max()), max_abs_pi_vs_reference=float(np.abs(p - z['pi']).max()),
                           max_rel_elbo_vs_reference=float(np.max(np.abs(np.array([l[0] for l in L[:13]]) - z['Li'][:len(L[:13])]) / np.abs(z['Li'][:len(L[:13])]))),
                           labels_equal=bool(np.array_equal(g.argmax(1), z['labels'])))
    api.set_precision(default)
    # device-resident: the same EM loop on CUDA tensors through the batch API (float32 kernels + float64 finish)
    vb = VbxBatch([T], fea.shape[1], S, device=dev)
    vb.set_option('gemm', 1)
    fea_d = torch.from_numpy(fea.astype(np.float32)).to(dev)
    phi_d = torch.from_numpy(Phi.astype(np.float32)).to(dev)
    q_d = torch.zeros((T, vb.S), dtype=torch.float32, device=dev)
    g_d = torch.empty_like(q_d)
    q_d[:, :S] = torch.from_numpy(q.astype(np.float32)).to(dev)
    p_d = torch.zeros((1, vb.S), dtype=torch.float32, device=dev)
    rho_d = torch.empty_like(fea_d)
    obuf = vb.output_buffers(40)

    def resident_step():
        vb.prepare_scale(fea_d, phi_d, out=rho_d)
        g_d.copy_(q_d)
        p_d.zero_()
        p_d[0, :S] = 1.0 / S
        return vb.run(g_d, p_d, Fa=kw['Fa'], Fb=kw['Fb'], loopProb=kw['loopProb'], maxIters=40, epsilon=1e-6, buffers=obuf)

    evs = []
    l0 = None
    for i in range(3 + args.steps):                 # production configuration: no per-kernel events, the run replayed as a CUDA graph
        if i == 3:
            torch.cuda.synchronize()
            l0 = vb.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = resident_step()
        e1.record()
        if i >= 3:
            evs.append((e0, e1))
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, g_d, p_d, out, S)
    res_ms = float(np.median([a.elapsed_time(b) for a, b in evs]))
    n_steps = len(evs)
    launches = (vb.launches - l0) / n_steps
    vb.set_option('timing', 1)                       # kernel pass: direct launches with per-kernel events
    for i in range(2 + 5):
        if i == 2:
            torch.cuda.synchronize()
            vb.timings(reset=True)
        out = resident_step()
    torch.cuda.synchronize()
    timings = {k: (ms * n_steps / 5.0, n * n_steps / 5.0) for k, (ms, n) in vb.timings(reset=True).items()}
    vb.set_option('timing', 0)
    n_it = int(out['n_iters'][0].item())
    clocks = sampler.stop(t_all0, time.time())
    m = modes[default]
    kernels = {k: {'ms_per_step': v[0] / n_steps, 'launches_per_step': v[1] / n_steps} for k, v in timings.items() if v[1]}
    # the call is launch/latency bound: a roofline fraction against HBM is reported for completeness only
    peaks = load_peaks()
    alg_bytes = T * (4 * R_DIM + 4 * S + 2 * 4 * R_DIM * n_it)
    line = {
        'metric': METRIC, 'value': T / (res_ms / 1e3), 'unit': UNIT, 'n_gpus': 1, 'steps': n_steps, 'warmup': 3,
        'ms_per_step': res_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32 kernels + f64 finishing phase',
        'data': 'real: ES2005a x-vectors projected by the reference chain (fixture tests/golden/es2005a.npz)',
        'config': workload_config(w, wname, 1),
        'note': f'value = device-resident batch API (CUDA tensors in/out, {n_it} iterations until the epsilon stop); e2e = the drop-in VBx() '
                f'with host numpy arrays in and out, precision {default!r}; both modes listed under dropin',
        'iterations': n_it, 'reference_iterations': 13,
        'e2e': {'value': T / (m['warm_ms'] / 1e3), 'unit': UNIT, 'ms_per_step': m['warm_ms'], 'cold_ms': m['cold_ms'],
                'h2d_bytes_per_step': int(fea.nbytes + Phi.nbytes + q.nbytes), 'd2h_bytes_per_step': int(q.nbytes + 8 * S + 8 * 40),
                'api': f'vbx_b200.api.VBx (the reference signature), precision {default!r}, plan cached across calls (warm) / created inside (cold)'},
        'dropin': modes,
        'roofline': {'bound': 'hbm', 'kernel': 'whole call (latency bound: one recording cannot fill the GPU)', 'achieved': alg_bytes / (res_ms * 1e-3) / 1e9,
                     'peak': peaks[0], 'unit': 'GB/s', 'frac': alg_bytes / (res_ms * 1e-3) / 1e9 / peaks[0], 'traffic': None, 'peak_source': peaks[1]},
        'kernels': kernels, 'gpu_launches': launches * n_steps, 'gpu_launches_per_step': launches, 'clocks': clocks,
    }
    if not args.no_cpu_baseline:
        fn, kind, desc = cpu_vbx()
        tasks = [(fea, None, Phi, q, S, 40, kw['Fa'], kw['Fb'], kw['loopProb'], 1e-6)]
        walls, used = cpu_pool_run(tasks, 1, repeats=2, warmup=1)
        line['cpu_baseline'] = {'value': T / min(walls), 'unit': UNIT, 'cores': 1, 'kind': kind, 'wall_s': min(walls),
                                'sample': f'the same call on the same recording, one process (run_example.sh runs one); {desc}'}
    print(json.dumps(line), flush=True)


def load_peaks():
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        if 'hbm_gbs' in peaks:
            return float(peaks['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
    except Exception:
        pass
    return 6650.0, 'fallback 6.65 TB/s (B200_PROFILING.md)'


DUMP_BYTES, DUMP_GAMMA_BYTES = 60 << 20, 32 << 20         # 60 MiB of payload + .npy headers stay under 64 MB


def dump_outputs(directory, gamma, pi, out, S, trace=None):
    """Write what the last timed step returned to its caller as DIR/<name>.npy (float32 / float64), for comparing two
    builds output for output: pi [B,S], Li, n_iters, flags (and the batch ELBO trace) in full, and the responsibilities
    gamma [N,S] for a fixed, seeded sample of frames (rows of the packed array, row indices alongside): at most 32 MB
    of gamma and 64 MB in all."""
    import torch
    arrays = {'pi': pi[:, :S].float(), 'Li': out['Li'].double(), 'n_iters': out['n_iters'].double(),
              'flags': out['flags'].double()}
    if trace is not None:
        arrays['elbo_trace'] = torch.as_tensor(np.asarray(trace, dtype=np.float64))
    rest = sum(a.numel() * a.element_size() for a in arrays.values())
    if rest > DUMP_BYTES // 2:
        raise SystemExit(f'--dump-outputs: the per-recording outputs alone take {rest} bytes')
    N = gamma.shape[0]
    k = min(N, DUMP_GAMMA_BYTES // (4 * S), (DUMP_BYTES - rest) // (4 * S + 8))
    rows = np.sort(np.random.default_rng(0).choice(N, size=k, replace=False))
    arrays['gamma_sample'] = gamma[torch.from_numpy(rows).to(gamma.device), :S].float()
    arrays['gamma_sample_rows'] = torch.from_numpy(rows.astype(np.float64))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + '.npy'), a.cpu().numpy())


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='headline', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--fb-spl', type=int, default=0)
    ap.add_argument('--projection', type=int, default=0)
    ap.add_argument('--fb-classic', type=int, default=0, help='1 = normalise-every-frame forward-backward sweep (A/B against the look-ahead kernel)')
    ap.add_argument('--opt', action='append', default=[], help='name=value passed to vbx_set_option (A/B runs)')
    ap.add_argument('--parts', type=int, default=0, help='sub-batches on separate streams (vbx_b200/parts.py): 0 = auto, 1 = off')
    ap.add_argument('--fb-split', type=int, default=0, help='0 = auto, 1 = always, 2 = never: forward / backward sweeps on separate warps')
    ap.add_argument('--front', default='project', choices=['project', 'xvectors'],
                    help="what feeds the EM loop: 'project' = rho = X.V (the headline definition, SURVEY 8d); 'xvectors' = the "
                         "real-data chain vbx_prepare_xvectors (x-vector transform + PLDA projection, two tcgen05 passes)")
    ap.add_argument('--extra', default='', help='comma separated extra workloads to time (kernel-only) in the same run')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (the inputs are seeded: the same '
                         'arguments give the same inputs, so two builds can be compared output for output).  With '
                         'several ranks, rank 0 writes its own recordings (gamma, pi, Li, n_iters, flags) and the '
                         'batch-wide elbo_trace')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the device path (--impl b200)')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    w, wname = WORKLOADS[args.workload], args.workload
    if args.impl == 'reference':
        return run_reference(args, w, wname)
    if w.get('dropin'):
        return run_c1(args, w, wname)

    import torch
    import torch.distributed as dist
    from vbx_b200 import shard
    from vbx_b200.batch import VbxBatch
    from vbx_b200.host_pipeline import HostPipeline
    from vbx_b200.parts import make_batch, PartitionedBatch

    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the VB-HMM path has no CPU fallback; use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    device = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=device)

    def barrier():
        if world > 1:
            dist.barrier()

    def dbg(msg):
        if os.environ.get('VBX_BENCH_DEBUG'):
            print(f'[rank {rank}] {msg}', file=sys.stderr, flush=True)

    def time_workload(w, wname, steps, warmup, with_clocks):
        strong = bool(w.get('strong'))
        if strong:          # one fixed job, LPT-partitioned over the ranks (vbx_b200/shard.py)
            all_lengths = workload_lengths(w, seed=1000)
            mine = shard.partition(all_lengths, world)[rank]
            lengths = all_lengths[mine]
            data = make_device_shard(all_lengths, mine, w['S'], seed=17, device=device)
        else:               # every rank owns its own batch
            lengths = workload_lengths(w, seed=1000 + rank)
            data = make_device_batch(lengths, w['S'], seed=17 + rank, device=device)
        N = int(lengths.sum())
        dbg(f'{wname}: data on device, {len(lengths)} recordings, N={N}')
        def configure(b, timing):
            if args.fb_spl:
                b.set_option('fb_states_per_lane', args.fb_spl)
            if args.projection:
                b.set_option('projection', args.projection)
            if args.fb_classic:
                b.set_option('fb_classic', 1)
            for kv in args.opt:
                k, _, v = kv.partition('=')
                b.set_option(k, int(v))
            b.set_option('timing', int(timing))

        vb = make_batch(lengths, R_DIM, w['S'], device=device, parts=args.parts, fb_split=args.fb_split)
        partitioned = isinstance(vb, PartitionedBatch)
        # the timed region runs the production configuration (no per-kernel events; small batches replay the run as one CUDA
        # graph, large ones overlap two sub-batches on two streams); per-kernel CUDA events come from a separate pass below
        configure(vb, timing=False)
        in_library_collective = vb.attach_comm() if world > 1 else False
        S = vb.S
        rho = torch.empty((N, R_DIM), dtype=torch.float32, device=device)
        gamma = torch.zeros((N, S), dtype=torch.float32, device=device)
        pi = torch.empty((len(lengths), S), dtype=torch.float32, device=device)
        pi0 = torch.zeros(S, device=device)
        pi0[:w['S']] = 1.0 / w['S']
        trace = torch.zeros(2 * w['iters'], dtype=torch.float64, device=device)
        flush = None
        if N * R_DIM * 4 <= 2 * 126e6:
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)
        vb.n_states = None if w['S'] == S else torch.full((len(lengths),), w['S'], dtype=torch.int32, device=device)

        model = None
        if args.front == 'xvectors':       # synthetic model with the shapes of VBx/models/ResNet101_16kHz
            gen = torch.Generator(device='cpu').manual_seed(5)
            rnd = lambda *shape: torch.randn(*shape, generator=gen)
            q, _ = torch.linalg.qr(rnd(R_DIM, R_DIM))
            model = [t.to(device).contiguous() for t in (
                rnd(D_RAW) * 0.5, rnd(D_RAW, R_DIM) / D_RAW ** 0.5, rnd(R_DIM) * 0.05, rnd(R_DIM) * 0.02,
                q * (2.0 + 18.0 * torch.rand(R_DIM, generator=gen))[:, None])] + [data['Phi']]

        obuf = vb.output_buffers(w['iters'])       # fixed output tensors: the run can be replayed as a CUDA graph

        def step():
            if model is None:
                vb.prepare_project(data['X'], data['V'], data['Phi'], out=rho)
            else:
                vb.prepare_xvectors(data['X'], *model, out=rho)
            gamma[:, :w['S']].copy_(data['gamma0'])
            pi.copy_(pi0.expand_as(pi))
            out = vb.run(gamma, pi, Fa=w['Fa'], Fb=w['Fb'], loopProb=w['loopP'], maxIters=w['iters'], epsilon=-float('inf'),
                         buffers=obuf if vb is not None and hasattr(vb, 'children') is False else None)
            trace.copy_(vb.elbo_trace(out['Li']))      # the one collective of the path, inside the library (NCCL)
            return out

        # nvidia-smi needs up to a second before its first sample on a busy 8-GPU box: start it before the warm-up
        sampler = ClockSampler(local_rank) if (with_clocks and rank == 0) else None
        if sampler:
            sampler.start()
        for _ in range(warmup):
            if flush is not None:
                flush.zero_()
            step()
        torch.cuda.synchronize()
        dbg('warm-up done')
        vb.timings(reset=True)
        l0 = vb.launches
        if sampler:
            t_wait = time.time()
            while not sampler.lines and time.time() - t_wait < 3.0:      # first sample in hand before the timed region
                time.sleep(0.05)
        torch.cuda.synchronize()
        barrier()                      # every rank enters the timed region together
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        t_wall0 = time.time()
        for i in range(steps):
            if flush is not None:
                flush.zero_()
            evs[i][0].record()
            out = step()
            evs[i][1].record()
        torch.cuda.synchronize()
        barrier()
        t_wall1 = time.time()
        clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
        per_step = [a.elapsed_time(b) for a, b in evs]
        if os.environ.get('VBX_BENCH_DEBUG'):
            print(f'[rank {rank}] per-step ms: {[round(x, 3) for x in per_step]} wall {1e3 * (t_wall1 - t_wall0) / steps:.3f} ms/step', file=sys.stderr, flush=True)
        ms = sum(per_step) / steps
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            nt = torch.tensor([N], dtype=torch.float64, device=device)
            dist.all_reduce(nt)
            N_total = int(nt.item())
        else:
            N_total = N
        timings = vb.timings(reset=True)
        launches = (vb.launches - l0) / steps
        tr = trace.cpu().numpy()          # batch-wide ELBO trace of the last timed step (all ranks, in-library all-reduce)
        # ---- kernel pass: 3 steps with per-kernel CUDA events on ONE stream, direct launches ----
        gamma_keep, pi_keep, out_keep = gamma.clone(), pi.clone(), {k: v.clone() for k, v in out.items() if k in ('Li', 'n_iters', 'flags')}
        if partitioned:
            serial = VbxBatch(lengths, R_DIM, w['S'], device=device, fb_split=args.fb_split)
            configure(serial, timing=True)
            serial.n_states = vb.n_states
        else:
            serial = vb
            serial.set_option('timing', 1)
        whole_vb, vb = vb, serial
        for i in range(2 + 3):
            if i == 2:
                torch.cuda.synchronize()
                serial.timings(reset=True)
            if flush is not None:
                flush.zero_()
            step()
        torch.cuda.synchronize()
        timings = {k: (ms * steps / 3.0, n * steps / 3.0) for k, (ms, n) in serial.timings(reset=True).items()}
        vb = whole_vb
        if partitioned:
            serial.close()
        else:
            vb.set_option('timing', 0)
        gamma.copy_(gamma_keep)
        pi.copy_(pi_keep)
        out = dict(out, **out_keep)
        kernel_pass = ('separate pass of 3 steps with per-kernel CUDA events (one stream, direct launches); the timed region runs '
                       + ('two sub-batches on two streams, so the per-kernel times add up to more than ms_per_step' if partitioned else
                          'without events and, for small batches, as one CUDA graph launch per run'))
        assert np.all(np.isfinite(tr)), 'non-finite ELBO in the benchmark run'
        n_all = world * w['B'] if not strong else w['B']
        assert np.all(tr[w['iters']:] == n_all), (tr[w['iters']:], n_all)       # every recording of the job ran every iteration
        return dict(ms=ms, N=N, N_total=N_total, timings=timings, launches=launches, clocks=clocks, lengths=lengths,
                    data=data, vb=vb, S=S, out=out, steps=steps, strong=strong, trace=tr, gamma=gamma, pi=pi,
                    in_library_collective=bool(in_library_collective), partitioned=partitioned, kernel_pass=kernel_pass,
                    parts=len(vb.children) if partitioned else 1)

    def parity_sample(res, w, n_rec=3):
        """Size-true check inside the bench: a few recordings of THIS batch against the float64 C oracle (the checker)."""
        from oracle import c_oracle
        lens = res['lengths']
        offs = np.concatenate([[0], np.cumsum(lens)])
        pick = sorted(set([0, len(lens) // 2, len(lens) - 1]))[:n_rec]
        V0 = res['data']['V0'].double().cpu().numpy()
        Phi = res['data']['Phi'].double().cpu().numpy()
        worst = dict(gamma=0.0, pi=0.0, elbo=0.0)
        for b in pick:
            lo, hi = int(offs[b]), int(offs[b + 1])
            fea = res['data']['X'][lo:hi].double().cpu().numpy() @ V0
            g0 = res['data']['gamma0'][lo:hi].double().cpu().numpy()
            ref = c_oracle.vbx_oracle_batch(fea, Phi, np.array([0, hi - lo]), g0, np.full(w['S'], 1.0 / w['S']), w['Fa'], w['Fb'], w['loopP'],
                                            w['iters'], -np.inf)
            worst['gamma'] = max(worst['gamma'], float(np.abs(res['gamma'][lo:hi, :w['S']].double().cpu().numpy() - ref['gamma']).max()))
            worst['pi'] = max(worst['pi'], float(np.abs(res['pi'][b, :w['S']].double().cpu().numpy() - ref['pi'][0]).max()))
            worst['elbo'] = max(worst['elbo'], float(np.nanmax(np.abs(res['out']['Li'][b].cpu().numpy() - ref['Li'][0]) / np.abs(ref['Li'][0]))))
        return {'recordings_checked': len(pick), 'frames_checked': int(sum(lens[b] for b in pick)), 'iterations': w['iters'],
                'max_abs_gamma': worst['gamma'], 'max_abs_pi': worst['pi'], 'max_rel_elbo': worst['elbo'],
                'bar': 'gamma, pi <= 1e-4 abs; ELBO <= 1e-4 relative (north_star)',
                'ok': bool(worst['gamma'] <= 1e-4 and worst['pi'] <= 1e-4 and worst['elbo'] <= 1e-4),
                'checker': 'oracle/vbx_oracle_c.c (float64) on the projected inputs of the sampled recordings, same iteration count'}

    res = time_workload(w, wname, args.steps, args.warmup, with_clocks=True)
    dbg(f'timed region done: {res["ms"]:.3f} ms/step')
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res['gamma'], res['pi'], res['out'], w['S'], trace=res['trace'])
    ms, N, N_total = res['ms'], res['N'], res['N_total']
    value = N_total / (ms / 1e3)

    # ---- roofline of the dominant kernel (CUDA events recorded inside the C ABI on the launching stream) ----
    peak_gbs, peak_src = load_peaks()
    S = res['S']
    alg_bytes = {   # algorithmic bytes per frame per launch (DESIGN.md section 4)
        'project': 4 * D_RAW + 4 * R_DIM if args.front == 'project' else 4 * D_RAW + 3 * 4 * R_DIM,
        'mstep_partial': 4 * R_DIM + 4 * S,
        'loglik': 4 * R_DIM + 4 * S + 4,
        'forward_backward': 5 * 4 * S + 12,
    }
    per_kernel = {}
    for k, (tms, cnt) in res['timings'].items():
        if cnt:
            per_kernel[k] = {'ms_per_launch': tms / cnt, 'launches_per_step': cnt / res['steps'], 'ms_per_step': tms / res['steps']}
            if k in alg_bytes:
                per_kernel[k]['gbs'] = alg_bytes[k] * N / (tms / cnt * 1e-3) / 1e9
    dom = max((k for k in per_kernel if k in alg_bytes), key=lambda k: per_kernel[k]['ms_per_step'])
    roof = {'bound': 'hbm', 'kernel': dom, 'achieved': per_kernel[dom]['gbs'], 'peak': peak_gbs, 'unit': 'GB/s',
            'frac': per_kernel[dom]['gbs'] / peak_gbs, 'traffic': None, 'peak_source': peak_src,
            'algorithmic_bytes_per_launch': alg_bytes[dom] * N, 'avg_launch_ms': per_kernel[dom]['ms_per_launch'],
            'share_of_step': per_kernel[dom]['ms_per_step'] / ms}
    traffic_file = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(traffic_file):
        try:
            tr = json.load(open(traffic_file))
            if tr.get('workload') == wname and dom in tr.get('dram_bytes_per_launch', {}):
                roof['traffic'] = tr['dram_bytes_per_launch'][dom]
                roof['traffic_source'] = tr.get('source')
        except Exception:
            pass
    step_bytes = N * (4 * D_RAW + 4 * R_DIM + 4 * w['S'] + 2 * 4 * R_DIM * w['iters'])   # SURVEY 8(d): N*(1600+1024*iters) at S=16
    whole = {'algorithmic_bytes_per_step': step_bytes, 'achieved_gbs': step_bytes / (ms * 1e-3) / 1e9,
             'frac_of_peak': step_bytes / (ms * 1e-3) / 1e9 / peak_gbs, 'per': 'GPU (this rank\'s frames over the max-over-ranks step time)'}

    parity = None
    if rank == 0 and not args.no_parity and args.front == 'project':
        parity = parity_sample(res, w)
        dbg(f'parity sample: {parity}')

    # ---- end-to-end through the host-buffer API (pinned host inputs, H2D + D2H inside the timed region) ----
    e2e = None
    if not args.no_e2e and args.front == 'project':
        numa = {}
        with numa_affinity(local_rank, numa):       # pinned buffers + feeding thread on the GPU's NUMA node
            hp = HostPipeline(res['lengths'], D_RAW, R_DIM, w['S'], device=device,
                              n_chunks=int(os.environ['VBX_E2E_CHUNKS']) if os.environ.get('VBX_E2E_CHUNKS') else None)
            Xh = torch.empty((N, D_RAW), dtype=torch.float32).pin_memory()
            Gh = torch.empty((N, w['S']), dtype=torch.float32).pin_memory()
            Xh.copy_(res['data']['X'])
            Gh.copy_(res['data']['gamma0'])
            torch.cuda.synchronize()
            kw = dict(Fa=w['Fa'], Fb=w['Fb'], loopProb=w['loopP'], maxIters=w['iters'], epsilon=-float('inf'))
            for _ in range(2):
                hp.run(Xh, res['data']['V'], res['data']['Phi'], Gh, **kw)
            barrier()
            torch.cuda.synchronize()
            n_e2e = max(3, min(args.steps, 5))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n_e2e):
                o = hp.run(Xh, res['data']['V'], res['data']['Phi'], Gh, **kw)
            e1.record()
            torch.cuda.synchronize()
            barrier()
        ems = e0.elapsed_time(e1) / n_e2e
        if world > 1:
            t = torch.tensor([ems], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
        # parity of the two paths on the same data (device-resident vs host-pipelined)
        dmax = float((o['gamma'].to(device) - res['gamma'][:, :w['S']]).abs().max())
        h2d, d2h = hp.h2d_bytes, hp.d2h_bytes
        if world > 1:
            tb = torch.tensor([h2d, d2h], dtype=torch.float64, device=device)
            dist.all_reduce(tb)
            h2d, d2h = int(tb[0].item()), int(tb[1].item())
        e2e = {'value': N_total / (ems / 1e3), 'unit': UNIT, 'ms_per_step': ems, 'h2d_bytes_per_step': h2d,
               'd2h_bytes_per_step': d2h, 'chunks': hp.n_chunks, 'max_abs_gamma_diff_vs_resident': dmax, 'numa': numa or None,
               'api': 'vbx_b200.host_pipeline.HostPipeline.run (pinned host X, gamma0 -> gamma, pi, Li on the host)'}
        del Xh, Gh, hp
        dbg('e2e done')

    # ---- CPU baseline on this box's host cores (rank 0, N=1) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        n_rec = max(8, min(cores, 64))
        ws, scale, bnote = bounded(w)
        recs, V0, Phi = host_sample(ws, n_rec, seed=1)
        tasks = [(X, V0, Phi, g0, ws['S'], ws['iters'], ws['Fa'], ws['Fb'], ws['loopP'], -np.inf) for X, g0 in recs]
        dbg('cpu baseline ...')
        walls, used = cpu_pool_run(tasks, cores)
        frames = sum(x.shape[0] for x, _ in recs)
        fn, kind, desc = cpu_vbx()
        cpu = {'value': frames / min(walls) * scale, 'unit': UNIT, 'cores': used, 'kind': kind, 'wall_s': min(walls),
               'sample': f'{len(recs)} recordings of the workload ({frames} x-vectors, {ws["iters"]} iterations), one process per recording on '
                         f'{used} cores; {desc}{bnote}'}
        try:
            from oracle import c_oracle
            t0 = time.perf_counter()
            sub = recs[:8]
            fea = np.concatenate([x.astype(np.float64) @ V0 for x, _ in sub])
            g0 = np.concatenate([g for _, g in sub])
            offs = np.concatenate([[0], np.cumsum([x.shape[0] for x, _ in sub])])
            c_oracle.vbx_oracle_batch(fea, Phi, offs, g0, np.full(w['S'], 1.0 / w['S']), w['Fa'], w['Fb'], w['loopP'], ws['iters'], -np.inf)
            cpu['c_oracle_single_thread'] = {'value': fea.shape[0] / (time.perf_counter() - t0) * scale, 'unit': UNIT,
                                             'note': 'oracle/vbx_oracle_c.c (O(S) scaled recursion, float64), 1 thread, 8 recordings'}
        except Exception as ex:   # the C oracle is optional here
            cpu['c_oracle_single_thread'] = {'error': str(ex)}

    extra = {}
    for name in [x for x in args.extra.split(',') if x]:
        r2 = time_workload(WORKLOADS[name], name, max(3, args.steps // 2), 3, with_clocks=False)
        extra[name] = {'value': r2['N_total'] / (r2['ms'] / 1e3), 'unit': UNIT, 'ms_per_step': r2['ms'],
                       'config': workload_config(WORKLOADS[name], name, world),
                       'kernels_ms_per_step': {k: v[0] / r2['steps'] for k, v in r2['timings'].items() if v[1]}}

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong' if res['strong'] else 'weak', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic (seeded sticky-Markov speakers in PLDA space, SURVEY.md 8d; generated on the device)',
            'config': workload_config(w, wname, world),
            'target': {'north_star_x_vectors_per_s': 1e7, 'ratio': value / 1e7 / max(world, 1)},
            'roofline': roof, 'whole_step': whole, 'kernels': per_kernel, 'kernels_measured': res['kernel_pass'],
            'sub_batches_on_streams': res['parts'], 'gpu_launches': res['launches'] * args.steps,
            'gpu_launches_per_step': res['launches'], 'clocks': res['clocks'], 'e2e': e2e, 'cpu_baseline': cpu, 'parity': parity,
            'elbo_trace': {'sum_per_iteration': [float(x) for x in res['trace'][:w['iters']]], 'recordings': int(res['trace'][w['iters']]),
                           'collective': ('ncclAllReduce inside vbx_elbo_trace (communicator attached with vbx_attach_comm)' if res['in_library_collective']
                                          else 'single GPU: no collective')},
        }
        if args.front != 'project':
            line['note'] = 'front end = vbx_prepare_xvectors (x-vector transform + PLDA projection) instead of rho = X.V; not the headline definition'
        if extra:
            line['other_workloads'] = extra
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
