"""Throughput of the compiled (dim_x, dim_u) shapes that the bench.py workloads leave out (systems.NEW_SHAPES).

For each shape: 16,384 members of systems.ensemble_shape under the nominal config_shape model, one warm-up pass, then
three timed resident passes (device events, L2 flushed between passes, as bench.py times its headline).  Reports
trajectories/s, QP solves/s, the launch geometry (warps per SM), the fp64 fraction (bench.py's flop model on the device
counters over the m4q_fp64_fma_probe rate of this run), and the card name and power limit read in the same run.

    python tools/bench_shapes.py [--members 16384] [--passes 3] [--shapes 9,1 16,4] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def card():
    import torch
    q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q)


def measure(c, m, n, passes, warmup, flush, fp64_peak):
    import bench
    import mpc4quantum_b200 as m4q
    from mpc4quantum_b200 import _lib, systems
    cfg = systems.config_shape(c, m)
    ens, _ = systems.ensemble_shape(cfg, n)
    plan = m4q.ClosedLoopPlan(cfg['dim_u'], cfg['order'], cfg['X_targ'], cfg['U_targ'], cfg['clock'], cfg['model'],
                              cfg['Q'], cfg['R'], cfg['Qf'], cfg['sat'], cfg['du'], d=ens.d, lift_mode=ens.lift_mode,
                              warm_start=cfg['warm_start'], fid_target=cfg['target'], capacity=n)
    x0 = cfg['u0'] if cfg.get('kind') == 'process' else cfg['x0']      # gate synthesis carries the propagator
    x0_d = _lib.dev(np.ascontiguousarray(x0.reshape(1, -1)), np.complex128)
    H0_d, H1_d = _lib.dev(ens.H0, np.complex128), _lib.dev(ens.H1, np.complex128)

    def run():
        return plan.run(x0_d, H0_d, H1_d, n=n, x0_shared=True)
    for _ in range(warmup):
        run()
    total_ms, per, res = bench.timed(run, passes, flush, 1, None)
    counters, qp_count = res.counters.cpu().numpy(), res.qp_count.cpu().numpy()
    exit_codes = res.exit_code.cpu().numpy()
    flops, _ = bench.flop_model(cfg, counters, qp_count)
    ms = total_ms / passes
    geom = plan.launch_info(n)
    return {'shape': [c, m], 'name': cfg['name'], 'members': n, 'horizon': cfg['clock'].horizon,
            'n_steps': cfg['clock'].n_steps, 'order': cfg['order'], 'ms_per_pass': per,
            'trajectories_per_s': n / (ms * 1e-3), 'qp_solves_per_s': float(counters[:, 3].sum()) / (ms * 1e-3),
            'qp_solves_per_trajectory': float(counters[:, 3].sum()) / n, 'launch': geom,
            'warps_per_sm': geom['warps_per_cta'] * geom['ctas'] // 148 if geom['ctas'] >= 148 else geom['warps_per_cta'],
            'fp64_tflops': flops / (ms * 1e-3) / 1e12, 'fp64_frac': flops / (ms * 1e-3) / 1e12 / fp64_peak,
            'exit_codes': {str(k): int((exit_codes == k).sum()) for k in np.unique(exit_codes)},
            'fidelity_median': float(np.median(res.fidelity.cpu().numpy()))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--members', type=int, default=16384)
    ap.add_argument('--passes', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--shapes', nargs='*', default=None, help='c,m pairs (default: every shape of systems.NEW_SHAPES)')
    ap.add_argument('--out', default=None, help='also write the JSON here')
    args = ap.parse_args()
    import torch
    import bench
    from mpc4quantum_b200 import systems
    if not torch.cuda.is_available():
        raise SystemExit('bench_shapes.py measures on the GPU; no CUDA device is present')
    shapes = [tuple(int(v) for v in s.split(',')) for s in args.shapes] if args.shapes else list(systems.NEW_SHAPES)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')      # > 126 MB L2
    fp64_peak, _ = bench.fp64_probes(0)
    out = {'card': card(), 'fp64_fma_probe_tflops': fp64_peak, 'results': []}
    for c, m in shapes:
        r = measure(c, m, args.members, args.passes, args.warmup, flush, fp64_peak)
        out['results'].append(r)
        print(json.dumps(r), flush=True)
    out['card_after'] = card()
    text = json.dumps(out, indent=1)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')
    print(text)


if __name__ == '__main__':
    main()
