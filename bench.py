#!/usr/bin/env python
"""Benchmark of the closed-loop MPC hot path (BASELINE.json: closed-loop MPC trajectories/s over an ensemble of
perturbed transmon plants).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload transmon_h16] [--members-total 65536 | --members M]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...      # the CPU path (oracle port of the reference) on the host cores

One "step" = one pass of the whole closed loop (all MPC steps of mpc.py:128-304) over this rank's shard of the
ensemble.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the flop model behind `roofline`.

Scaling: the north_star's target is ONE 65,536-member ensemble at 1/2/4/8 GPUs, so the headline `value` is STRONG
scaling (`--members-total`, default 65,536: every rank takes 1/N of the same seeded ensemble); the weak-scaling number
(65,536 members per GPU, `--members`) is measured in the same run and reported under `extra.weak` when N > 1.
`extra.workloads` carries the other BASELINE configs (2, 4, the horizon sweep of 3, and 5 on 8 GPUs) measured the same
way on shorter runs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'closed-loop MPC trajectories/s'
UNIT = 'trajectories/s'
DUMP_SEED = 20220113        # member sample of --dump-outputs


# ----------------------------------------------------------------------------------------------------------
SYSTEM_NAMES = {'transmon': '3-level transmon', 'qubit': 'ideal qubit', 'crosstalk': 'two qubits with ZZ crosstalk',
                'not_gate': 'NOT-gate synthesis on the qubit process vector',
                'transmon_exact': '3-level transmon, exact-discretisation model'}


def workload(name, discretize=None):
    from mpc4quantum_b200 import systems
    if name.startswith('transmon_h') or name.startswith('transmon_o2_h') or name.startswith('transmon_models_h'):
        order = 2 if name.startswith('transmon_o2_h') else 1
        H = int(name.split('_h')[-1])
        cfg = systems.config_transmon(order, horizon=H, n_steps=20, discretize=discretize)
        # transmon_models_hH: every member also controls with its own perturbed MODEL (discretised per member)
        cfg['per_member_models'] = name.startswith('transmon_models_h')
        return cfg, systems.ensemble_transmon
    if name.startswith('transmon_exact_h'):    # exact-discretisation model mode (expm + Frechet derivative per stage)
        return systems.config_transmon_exact(horizon=int(name.split('_h')[-1]), n_steps=20), systems.ensemble_transmon
    if name == 'qubit':
        return systems.config_qubit(1, discretize=discretize), systems.ensemble_qubit
    if name == 'crosstalk':
        return systems.config_crosstalk(0.0, discretize=discretize), systems.ensemble_crosstalk
    if name == 'not_gate':      # gate synthesis on process vectors (c = 16, m = 1, H = 15, S = 50)
        return systems.config_not_gate(1, discretize=discretize), systems.ensemble_not_gate
    raise SystemExit('unknown workload %s' % name)


def flop_model(cfg, counters, qp_count):
    """Algorithmic real flops of a batch of trajectories (SURVEY.md section 8d) from the device counters.

    counters [n, 4] = ADMM iterations, Riccati factorisations, polish rounds, QP solves.
    """
    exact = hasattr(cfg['model'], 'generators')
    c = cfg['model'].dim_x if exact else cfg['model'].A.shape[0]
    n, m = 2 * c, cfg['dim_u']
    p = m if exact else cfg['model'].A.shape[1] // c - 1
    H, S = cfg['clock'].horizon, cfg['clock'].n_steps
    d = cfg['experiment'].H0.shape[0]
    F_lin = H * (12 * p * c * c + 4 * p * c * m + 4 * c * m)
    if exact:   # per stage: expm by 16 Horner + ~3 squaring products (8 c^3 each), ~22 Taylor terms of (1 + 2m) complex
        #           mat-vecs for the Frechet vectors (term count depends on the generator norm; 22 at ||G dt|| ~ 1.5)
        F_lin = H * (19 * 8 * c ** 3 + 22 * (1 + 2 * m) * 8 * c * c)
    F_fac = H * (4 * n ** 3 + 6 * n * n * m + 2 * n * m * m + m ** 3)
    F_it = H * (4 * n * n + 8 * n * m)
    F_ls = 6 * (2 * c * (H + 1) + 2 * m * H)
    F_pl = 8 * d ** 3 * (18 + 2)
    admm, factor, polish, solves = [counters[:, i].astype(np.float64).sum() for i in range(4)]
    ls_calls = float(qp_count[:, :2].sum()) if cfg['warm_start'] else solves
    total = solves * F_lin + factor * F_fac + (admm + 2 * polish) * F_it + ls_calls * F_ls + counters.shape[0] * S * F_pl
    return total, dict(F_lin=F_lin, F_fac=F_fac, F_it=F_it, F_ls=F_ls, F_pl=F_pl)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled while the timed region runs (B200_PROFILING.md)."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.rows = []

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(',')]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = [float(r[0]) for r in self.rows]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [nm for i, nm in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(self.rows[0][1]), 'reasons': reasons,
                'power_w_max': max(float(r[2]) for r in self.rows), 'samples': len(self.rows)}


# ----------------------------------------------------------------------------------------------------------
# CPU path: the oracle port of the reference loop (oracle/restate.py), one process per core
# ----------------------------------------------------------------------------------------------------------
def _cpu_member(job):
    name, k, n_total = job
    os.environ['OMP_NUM_THREADS'] = '1'
    from oracle import restate as rs
    cfg, maker = workload(name, discretize=rs.taylor_discretize)
    ens, _ = maker(n_total, lo=k, hi=k + 1)      # member k of the seeded ensemble, drawn alone
    mem = ens.member(0)
    lift, proj = (rs.lift_coupled, rs.proj_coupled) if cfg.get('kind') == 'coupled' else (rs.lift_identity, rs.lift_identity)
    plant = rs.ProcessPlant(mem.H0, mem.H1_list) if cfg.get('kind') == 'process' else \
        rs.ExpmPlant(mem.H0, mem.H1_list, lift, proj)
    stats = {}
    A_full = getattr(cfg['model'], 'A', None)
    if cfg.get('per_member_models'):
        from mpc4quantum_b200 import systems
        L, _ = systems.transmon_model_liouvillians(n_total, lo=k, hi=k + 1)
        A_full = rs.taylor_discretize(list(L[0]), cfg['clock'].dt, cfg['order'])
    exact = rs.ExactModel(list(cfg['model'].generators), cfg['clock'].dt) if cfg['name'] == 'transmon_exact' else None
    xs, us, ec = rs.mpc_loop(cfg['x0'], cfg['dim_u'], cfg['order'], cfg['X_targ'], cfg['U_targ'], cfg['clock'].dt,
                             cfg['clock'].horizon, cfg['clock'].n_steps, plant, A_full, cfg['Q'], cfg['R'],
                             cfg['Qf'], cfg['sat'], cfg['du'], warm_start=cfg['warm_start'],
                             measure_freq=cfg['clock'].measure_freq, stats=stats, model=exact)
    return float(np.real(np.vdot(cfg['target'], xs[:, -1]))), int(sum(stats['qp_per_step']))


def cpu_pass(name, members, n_total, pool):
    t0 = time.perf_counter()
    res = pool.map(_cpu_member, [(name, k, n_total) for k in members])
    dt = time.perf_counter() - t0
    return dt, res


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_reference_arm(args):
    """`--impl reference`: the reference's CPU algorithm (oracle port: reference loop semantics with exact QP and
    expm plant leaves, see oracle/restate.py) on all host cores.  Each step = a bounded sample of the workload."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = host_cores()
    per_step = max(cores, 8)
    n_total = args.members_total
    with mp.get_context('spawn').Pool(cores) as pool:
        cpu_pass(args.workload, range(min(cores, 4)), n_total, pool)          # import / page-in warm-up
        for w in range(args.warmup):
            cpu_pass(args.workload, range(w * per_step, (w + 1) * per_step), n_total, pool)
        t_total, qps = 0.0, 0
        for s in range(args.steps):
            dt, res = cpu_pass(args.workload, range(s * per_step, (s + 1) * per_step), n_total, pool)
            t_total += dt
            qps += sum(r[1] for r in res)
    value = args.steps * per_step / t_total
    sample = '%d members per step (first members of the same seeded ensemble), %d steps' % (per_step, args.steps)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * t_total / args.steps, 'higher_is_better': True,
        'scaling': 'weak' if args.members is not None else 'strong',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': '%s, one ensemble of %d perturbed plants (seed 20220113)' % (args.workload, n_total),
                   'members_total': n_total,
                   'note': 'CPU arm times a bounded sample and reports trajectories/s of the host'},
        'qp_solves_per_s': qps / t_total,
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample,
                         'what': 'reference loop semantics (mpc.py:128-304) restated in numpy with exact active-set QP '
                                 'and scipy expm plant leaves; cvxpy/OSQP/qutip are not installable offline'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------
class Runner:
    """One workload on this rank's shard: plan, resident inputs, pinned host inputs, timed passes."""

    def __init__(self, name, n_total, rank, world, admm_first=False):
        import torch
        import mpc4quantum_b200 as m4q
        from mpc4quantum_b200 import _lib, systems
        from mpc4quantum_b200.ensemble import shard_bounds
        self.torch, self.m4q, self.name = torch, m4q, name
        self.cfg, maker = workload(name)
        cfg = self.cfg
        self.n_total, self.world = n_total, world
        lo, hi = shard_bounds(n_total, rank, world)
        self.lo, self.n = lo, hi - lo
        self.ens, _ = maker(n_total, lo=lo, hi=hi)           # this rank's block of the seeded draw, nothing else
        model = cfg['model']
        if cfg.get('per_member_models'):
            model = systems.ensemble_transmon_models(n_total, order=cfg['order'], lo=lo, hi=hi)[0]
        self.model = model
        self.margs = (cfg['dim_u'], cfg['order'], cfg['X_targ'], cfg['U_targ'], cfg['clock'], model, cfg['Q'], cfg['R'],
                      cfg['Qf'], cfg['sat'], cfg['du'])
        self.plan = m4q.ClosedLoopPlan(*self.margs, d=self.ens.d, lift_mode=self.ens.lift_mode,
                                       warm_start=cfg['warm_start'], fid_target=cfg['target'], capacity=self.n,
                                       settings=_lib.qp_settings(admm_first=int(admm_first)) if admm_first else None)
        self.geom = self.plan.launch_info(self.n)
        x0_plant = cfg['u0'] if cfg.get('kind') == 'process' else cfg['x0']     # gate synthesis: the propagator itself
        self.x0_host = np.ascontiguousarray(x0_plant.reshape(-1))
        self.H0_d = _lib.dev(self.ens.H0, np.complex128)
        self.H1_d = _lib.dev(self.ens.H1, np.complex128)
        self.x0_d = _lib.dev(self.x0_host.reshape(1, -1), np.complex128)
        # the public API takes the experiment with HOST arrays: pinned, so that the copies inside the timed e2e pass run
        # at PCIe speed (mpc_ensemble moves them with torch; results come back through the plan's pinned buffers)
        self.H0_pin = torch.from_numpy(np.ascontiguousarray(self.ens.H0)).pin_memory()
        self.H1_pin = torch.from_numpy(np.ascontiguousarray(self.ens.H1)).pin_memory()
        self.ens_host = m4q.EnsembleQExperiment(self.H0_pin, self.H1_pin, self.ens.kind)
        self.hist = torch.zeros(256, dtype=torch.int64, device='cuda')

    def resident_pass(self, reduce=True):
        from mpc4quantum_b200.ensemble import fidelity_histogram, allreduce_histogram
        res = self.plan.run(self.x0_d, self.H0_d, self.H1_d, n=self.n, x0_shared=True)
        if reduce:
            self.hist.zero_()
            fidelity_histogram(res.fidelity, 0.0, 1.0, 256, self.hist)
            if self.world > 1:
                allreduce_histogram(self.hist)
        return res

    def outputs(self, res, max_members=4096, budget=60 << 20):
        """What a resident pass hands its caller, as float64 host arrays: every field of the EnsembleResult (complex
        arrays with a trailing (real, imag) axis) and the fidelity histogram.  Per-member arrays are taken at a fixed,
        seeded sample of this rank's members, whose global indices are `members`, so that the whole stays within
        `budget` bytes at any ensemble size while two builds can be compared member for member."""
        torch = self.torch
        fields = {k: getattr(res, k) for k in res.__slots__ if getattr(res, k) is not None}
        per_member = 8 + sum(8 * (2 if v.is_complex() else 1) * v[0].numel() for v in fields.values())
        k = min(self.n, max_members, (budget - 8 * self.hist.numel()) // per_member)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(self.n, k, replace=False))
        sel = torch.from_numpy(idx).to(self.hist.device)
        out = {'members': (self.lo + idx).astype(np.float64), 'fidelity_histogram': self.hist.double().cpu().numpy()}
        for name, v in fields.items():
            v = v.index_select(0, sel)
            out[name] = (torch.view_as_real(v) if v.is_complex() else v).double().cpu().numpy()
        return out

    def e2e_pass(self):
        """The call a user makes: host buffers in, numpy results (xs, us, fidelity, exit codes, counters) out."""
        cfg = self.cfg
        return self.m4q.mpc_ensemble(self.x0_host, *self.margs[:5], self.ens_host, *self.margs[5:],
                                     warm_start=cfg['warm_start'], fid_target=cfg['target'], plan=self.plan)

    def e2e_bytes(self, res):
        h2d = self.H0_pin.numel() * 16 + self.H1_pin.numel() * 16 + self.x0_host.size * 16
        d2h = sum(getattr(res, k).nbytes for k in res.__slots__ if getattr(res, k) is not None)
        return int(h2d), int(d2h)


def timed(fn, steps, flush, world, dist):
    """Device time of `steps` passes, L2 flushed between passes (flush not timed); max over ranks of the sum."""
    import torch

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
    total_ms, per, last = 0.0, [], None
    for _ in range(steps):
        flush.fill_(1)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = fn()
        e1.record()
        sync_all()
        per.append(e0.elapsed_time(e1))
        total_ms += per[-1]
    t = torch.tensor([total_ms], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), per, last


def measure(run, steps, warmup, flush, world, dist, fp64_peak=None, e2e=True, kernel_passes=None, keep_outputs=False):
    """value / kernel time / roofline of one Runner; returns a dict (with keep_outputs, 'outputs' holds
    Runner.outputs() of the last timed pass)."""
    import torch
    for _ in range(warmup):
        run.resident_pass()
    total_ms, _, last = timed(run.resident_pass, steps, flush, world, dist)
    outputs = run.outputs(last) if keep_outputs else None      # before the next pass overwrites the plan's buffers
    res = run.resident_pass()
    torch.cuda.synchronize()
    counters = res.counters.cpu().numpy()
    qp_count = res.qp_count.cpu().numpy()
    exit_codes = res.exit_code.cpu().numpy()
    fid = res.fidelity.cpu().numpy()
    kern = []
    for _ in range(kernel_passes or max(2, min(steps, 3))):          # the dominant kernel alone (no histogram / all-reduce)
        flush.fill_(1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run.resident_pass(reduce=False)
        e1.record()
        torch.cuda.synchronize()
        kern.append(e0.elapsed_time(e1))
    kernel_ms = float(np.mean(kern))
    flops, per_unit = flop_model(run.cfg, counters, qp_count)
    qp_total = float(counters[:, 3].sum())
    t = torch.tensor([qp_total, flops, float((exit_codes != 0).sum())], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(t)
    qp_all, flops_all, bad_all = t.tolist()
    out = dict(value=run.n_total * steps / (total_ms * 1e-3), ms_per_step=total_ms / steps, kernel_ms=kernel_ms,
               flops=flops, per_unit=per_unit, qp_total=qp_total, qp_all=qp_all, counters=counters, qp_count=qp_count,
               exit_codes=exit_codes, fid=fid, members_not_exit0_all_ranks=int(bad_all),
               achieved_tflops=flops / (kernel_ms * 1e-3) / 1e12, outputs=outputs)
    if fp64_peak:
        out['frac'] = out['achieved_tflops'] / fp64_peak
    if e2e:
        r = run.e2e_pass()                                  # untimed: first use of the pinned staging buffers
        e2e_steps = max(2, min(steps, 3))
        e2e_ms, per, _ = timed(run.e2e_pass, e2e_steps, flush, world, dist)
        h2d, d2h = run.e2e_bytes(r)
        out['e2e'] = {'value': run.n_total * e2e_steps / (e2e_ms * 1e-3), 'unit': UNIT, 'ms_per_pass': per,
                      'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                      'api': 'mpc4quantum_b200.mpc_ensemble(host arrays) -> numpy xs, us, fidelity, exit codes, counters'}
    return out


def summary(m, run):
    """Compact record of a secondary workload for extra.workloads."""
    ec = m['exit_codes']
    return {'members_total': run.n_total, 'value': m['value'], 'unit': UNIT, 'ms_per_step': m['ms_per_step'],
            'qp_solves_per_s': m['qp_all'] / (m['ms_per_step'] * 1e-3),
            'qp_solves_per_trajectory': m['qp_total'] / run.n, 'fp64_frac': m.get('frac'),
            'admm_iterations_per_qp': float(m['counters'][:, 0].sum() / max(m['qp_total'], 1)),
            'factorizations_per_qp': float(m['counters'][:, 1].sum() / max(m['qp_total'], 1)),
            'exit_codes_rank0': {str(k): int((ec == k).sum()) for k in np.unique(ec)},
            'members_not_exit0_all_ranks': m['members_not_exit0_all_ranks'],
            'fidelity_median_rank0': float(np.median(m['fid'])), 'launch': run.geom,
            'horizon': run.cfg['clock'].horizon, 'order': run.cfg['order']}


def fp64_probes(local):
    import torch
    from mpc4quantum_b200 import _lib
    scratch = torch.zeros(8, dtype=torch.float64, device='cuda')
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    ctas, iters = sms * 8, 1 << 16
    best = [0.0, 0.0]
    for which, (fn, it, per) in enumerate(((_lib.lib().m4q_fp64_fma_probe, iters, 2.0 * 16 * 256),
                                           (_lib.lib().m4q_fp64_dmma_probe, iters >> 2, 512.0 * 8 * 8))):
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(fn(ctas, it, _lib.ptr(scratch), _lib.stream_ptr()))
            e1.record()
            torch.cuda.synchronize()
            best[which] = max(best[which], per * it * ctas / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='transmon_h16')
    ap.add_argument('--members-total', type=int, default=None,
                    help='size of ONE ensemble split over the GPUs (strong scaling; default 65536)')
    ap.add_argument('--members', type=int, default=None,
                    help='ensemble members PER GPU (weak scaling); overrides --members-total for the headline')
    ap.add_argument('--cpu-seconds', type=float, default=20.0, help='budget of the cpu_baseline leg')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-extra', action='store_true', help='skip extra.weak / extra.workloads')
    ap.add_argument('--admm-first', action='store_true',
                    help='always run an ADMM block before the active-set rounds (m4q_qp_settings.admm_first)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed pass computed as DIR/<name>.npy: a seeded sample of the members of '
                         'rank 0 (with --gpus N > 1 only the first 1/N of the ensemble), their global indices in '
                         'members.npy, and the fidelity histogram of the whole ensemble')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs is not None and args.impl != 'b200':
        ap.error('--dump-outputs records the outputs of the b200 path')
    weak = args.members is not None
    if weak:
        args.members_total = args.members * args.gpus
    elif args.members_total is None:
        args.members_total = 65536
    if args.impl == 'reference':
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    assert world == args.gpus, 'launch with torchrun --nproc-per-node %d' % args.gpus

    n_total = args.members_total
    run = Runner(args.workload, n_total, rank, world, args.admm_first)
    cfg, n = run.cfg, run.n
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')      # > 126 MB L2
    S = cfg['clock'].n_steps

    fp64_peak, dmma_peak = fp64_probes(local)
    for _ in range(args.warmup):
        run.resident_pass()
    sampler = ClockSampler(local)
    sampler.start()
    dump = args.dump_outputs is not None and rank == 0
    m = measure(run, args.steps, 0, flush, world, dist, fp64_peak, keep_outputs=dump)
    sampler.stop_flag.set()
    sampler.join()
    if dump:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in m['outputs'].items():
            np.save(os.path.join(args.dump_outputs, name + '.npy'), arr)
    counters, qp_count, exit_codes, fid = m['counters'], m['qp_count'], m['exit_codes'], m['fid']
    res_bytes = m['e2e']['h2d_bytes_per_step'] + m['e2e']['d2h_bytes_per_step']

    # DRAM traffic of the dominant kernel: from the committed ncu capture (profiles/), scaled to this launch's members
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, 'profiles', 'r2b_ncu_traffic.json')) as fh:
            tr = json.load(fh)
        if args.workload == 'transmon_h16':
            traffic = (tr['dram_bytes_read'] + tr['dram_bytes_write']) * n / tr['members']
            traffic_src = ('ncu dram__bytes_read.sum + dram__bytes_write.sum of one %d-member launch '
                           '(profiles/r2b_ncu_traffic.json), scaled by members' % tr['members'])
    except (OSError, KeyError, ValueError):
        pass
    c_model = cfg['model'].dim_x if hasattr(cfg['model'], 'generators') else cfg['model'].A.shape[0]
    line = {
        'metric': METRIC, 'value': m['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': m['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak' if weak else 'strong',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': '%s: %s (c=%d, m=%d), horizon %d, %d MPC steps, one ensemble of %d perturbed plants '
                               '(seed 20220113) %s, tight QP mode (%s)' % (
                                   args.workload, SYSTEM_NAMES.get(cfg['name'], cfg['name']), c_model, cfg['dim_u'],
                                   cfg['clock'].horizon, S, n_total,
                                   ('= %d per GPU' % args.members) if weak else 'split over the GPUs',
                                   'ADMM block first' if args.admm_first else 'warm active set first, ADMM fallback'),
                   'members_total': n_total, 'members_this_rank': n,
                   'l2': 'flushed between timed passes (256 MB write, untimed)', 'launch': run.geom},
        'qp_solves_per_s': m['qp_all'] / (m['ms_per_step'] * 1e-3),
        'qp_solves_per_trajectory': m['qp_total'] / n,
        'admm_iterations_per_qp': float(counters[:, 0].sum() / max(m['qp_total'], 1)),
        'factorizations_per_qp': float(counters[:, 1].sum() / max(m['qp_total'], 1)),
        'exit_codes': {str(k): int((exit_codes == k).sum()) for k in np.unique(exit_codes)},
        'members_not_exit0_all_ranks': m['members_not_exit0_all_ranks'],
        'fidelity': {'min': float(fid.min()), 'median': float(np.median(fid)), 'max': float(fid.max()),
                     'convention': '<psi|rho|psi> (fidelity_sqrt = 0); qutip.fidelity is its square root'},
        'e2e': m['e2e'],
        'gpu_launches': 3 * args.steps,     # build_tables + mpc_kernel + hist_kernel per pass
        'roofline': {'bound': 'fp64', 'achieved': m['achieved_tflops'], 'peak': fp64_peak, 'unit': 'TFLOP/s',
                     'frac': m['frac'], 'traffic': traffic, 'traffic_source': traffic_src,
                     'peak_source': 'm4q_fp64_fma_probe measured in this run (MEASURED_PEAKS.json has no fp64 figure)',
                     'dmma_probe_tflops': dmma_peak,
                     'kernel': 'mpc_kernel', 'kernel_ms': m['kernel_ms'], 'flops_per_launch': m['flops'],
                     'flops_per_trajectory': m['flops'] / n, 'flop_model': m['per_unit'],
                     'hbm': {'algorithmic_bytes': int(res_bytes),
                             'achieved_gbs': res_bytes / (m['kernel_ms'] * 1e-3) / 1e9}},
        'clocks': sampler.summary(),
    }

    # ---- extra: the weak-scaling number beside the strong one, and the other BASELINE configs
    extra = {}
    if not args.no_extra:
        short = dict(steps=2, warmup=2, flush=flush, world=world, dist=dist, fp64_peak=fp64_peak, e2e=False)
        if world > 1 and not weak:
            del run
            torch.cuda.empty_cache()
            rw = Runner(args.workload, 65536 * world, rank, world, args.admm_first)
            mw = measure(rw, **short)
            extra['weak'] = dict(summary(mw, rw), scaling='weak', members_per_gpu=65536)
            del rw
            torch.cuda.empty_cache()
        if args.workload == 'transmon_h16':
            wl = {}
            todo = [('qubit', 4096, 'BASELINE config 2'), ('crosstalk', 65536, 'BASELINE config 4')] + \
                   [('transmon_h%d' % h, 16384, 'BASELINE config 3 horizon sweep, order-1 model') for h in (10, 20, 50)] + \
                   [('transmon_h100', 592, 'BASELINE config 3 horizon sweep, order-1 model: from the fourth step on every QP '
                                            'goes through the pivoted KKT solve (interior point + polish), ~300 block '
                                            'eliminations per trajectory; four members per SM, 1 timed pass')] + \
                   [('transmon_o2_h100', 16384, 'config 3 horizon sweep, order-2 model')]
            if world == 8:
                todo.append(('transmon_h16', 1 << 20, 'BASELINE config 5: 1 M perturbed transmons on 8 GPUs, '
                                                     'fidelity histogram all-reduced over NCCL'))
            for name, nt, what in todo:
                t_wl = time.time()
                try:
                    rx_ = Runner(name, nt, rank, world)
                    key = name if nt != (1 << 20) else 'transmon_h16_1M'
                    kw_ = dict(short, steps=1, warmup=1, kernel_passes=1) if name == 'transmon_h100' else short
                    wl[key] = dict(summary(measure(rx_, **kw_), rx_), what=what)
                    del rx_
                except Exception as e:                      # a secondary workload never takes the headline down
                    wl[name] = {'error': repr(e)[:200], 'what': what}
                torch.cuda.empty_cache()
                if rank == 0:
                    print('[bench] extra workload %s (%d members): %.1f s' % (name, nt, time.time() - t_wl), file=sys.stderr)
            extra['workloads'] = wl
    line['extra'] = extra

    if rank == 0 and not args.no_cpu and world == 1:
        import multiprocessing as mp
        cores = host_cores()
        with mp.get_context('spawn').Pool(cores) as pool:
            cpu_pass(args.workload, range(min(cores, 4)), n_total, pool)
            t0 = time.perf_counter()
            k_done, qps, cpu_fid = 0, 0, []
            while time.perf_counter() - t0 < args.cpu_seconds and k_done < n:
                dt, r = cpu_pass(args.workload, range(k_done, k_done + cores), n_total, pool)
                cpu_fid += [x[0] for x in r]
                qps += sum(x[1] for x in r)
                k_done += cores
            cpu_t = time.perf_counter() - t0
        # BASELINE.md section 4.3 (i): one process, one thread, a few members -> the per-core figure measured directly
        single = None
        try:
            from threadpoolctl import threadpool_limits
            with threadpool_limits(limits=1):
                t1 = time.perf_counter()
                rs_ = [_cpu_member((args.workload, k, n_total)) for k in range(3)]
                t_single = time.perf_counter() - t1
            single = {'members': 3, 'threads': 1, 'trajectories_per_s': 3 / t_single,
                      'qp_solves_per_s': sum(x[1] for x in rs_) / t_single}
        except Exception as e:                                  # the multi-process figure above does not depend on this
            single = {'error': repr(e)[:120]}
        cpu_model = ''
        try:
            with open('/proc/cpuinfo') as fh:
                cpu_model = next((ln.split(':', 1)[1].strip() for ln in fh if ln.startswith('model name')), '')
        except OSError:
            pass
        line['cpu_baseline'] = {
            'host': {'cpu_count': os.cpu_count(), 'affinity': cores, 'model': cpu_model},
            'single_process_single_thread': single,
            'value': k_done / cpu_t, 'unit': UNIT, 'cores': cores, 'kind': 'port',
            'sample': 'first %d members of the same ensemble, %.1f s' % (k_done, cpu_t),
            'qp_solves_per_s': qps / cpu_t,
            'per_core': {'trajectories_per_s': k_done / cpu_t / cores, 'qp_solves_per_s': qps / cpu_t / cores},
            'extrapolated_seconds_for_the_workload': n_total / (k_done / cpu_t),
            'calibration': 'port vs the reference mpc() through the shim on the build box: profiles/r2_cpu_calibration.json',
            'max_abs_fidelity_gap_vs_gpu': float(np.abs(np.array(cpu_fid) - fid[:k_done]).max())}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
