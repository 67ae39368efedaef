"""Compare two `bench.py --dump-outputs` directories output for output.

    python tools/compare_dumps.py OLD_DIR NEW_DIR [--us-tol 1e-8] [--fid-tol 1e-9]

Exit codes, steps done and QP counts must be identical; controls (`us`) must agree to --us-tol and fidelities to
--fid-tol (absolute).  Every other array is reported with its largest difference.  Members that differ are listed by
their global index (`members.npy`).  Exits 1 if a check fails.
"""
import argparse
import os
import sys

import numpy as np

EXACT = ('exit_code', 'steps_done', 'qp_count', 'members')


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith('.npy')}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('old')
    ap.add_argument('new')
    ap.add_argument('--us-tol', type=float, default=1e-8)
    ap.add_argument('--fid-tol', type=float, default=1e-9)
    a = ap.parse_args()
    old, new = load(a.old), load(a.new)
    ok = True
    if sorted(old) != sorted(new):
        print('array sets differ: %s vs %s' % (sorted(old), sorted(new)))
        ok = False
    members = old.get('members')
    for name in sorted(set(old) & set(new)):
        x, y = old[name], new[name]
        if x.shape != y.shape:
            print('%-16s shape %s vs %s' % (name, x.shape, y.shape))
            ok = False
            continue
        diff = np.abs(x.astype(np.float64) - y.astype(np.float64))
        both_nan = np.isnan(x) & np.isnan(y) if x.dtype.kind == 'f' else np.zeros(x.shape, bool)
        diff[both_nan] = 0.0
        dmax = float(diff.max()) if diff.size else 0.0
        tol = 0.0 if name in EXACT else a.us_tol if name == 'us' else a.fid_tol if name.startswith('fidelity') else None
        status = '' if tol is None else ('ok' if dmax <= tol else 'FAIL')
        ok &= status != 'FAIL'
        print('%-16s max |diff| %.3e %s' % (name, dmax, status))
        if status == 'FAIL' and members is not None and x.ndim >= 1 and x.shape[0] == len(members):
            bad = np.nonzero(diff.reshape(len(members), -1).max(axis=1) > tol)[0]
            print('    members that differ (%d): %s' % (len(bad), members[bad[:20]].astype(np.int64).tolist()))
    print('OK' if ok else 'FAILED')
    return 0 if ok else 1


if __name__ == '__main__':
    sys.exit(main())
