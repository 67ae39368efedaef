"""The horizon QP -- API of mpc4quantum/optimize.py.

``quad_program`` (optimize.py:12-60) states a box-constrained LTV tracking QP in cvxpy and hands it to OSQP.
Here the same problem is solved on the device by ``m4q_qp_admm_batched``: ADMM on the control box whose inner
linear system is a time-varying Riccati recursion in shared memory, followed (tight mode, the default) by an
active-set polish that certifies the KKT conditions.
"""
import numpy as np

from . import _lib


class QPInfo:
    """Stands in for the cvxpy problem object returned as the 4th value (optimize.py:60)."""

    def __init__(self, status, value, admm_iterations, factorizations):
        self.status = {0: 'optimal', 2: 'optimal_inaccurate', 3: 'infeasible_or_unbounded'}.get(int(status), 'unknown')
        self.status_code = int(status)
        self.value = value
        self.admm_iterations = int(admm_iterations)
        self.factorizations = int(factorizations)


def quad_program_batched(x_init, X_bm, U_bm, Q_ls, R_ls, A_ls, B_ls, Delta_ls, u_prev=None, sat=None, du=None,
                         settings=None):
    """Batched device front end; every argument carries a leading instance axis.

    x_init [N,c], X_bm [N,c,H+1], U_bm [N,m,H], Q_ls [N,H+1,c,c], R_ls [N,H,m,m], A_ls [N,H,c,c], B_ls [N,H,c,m],
    Delta_ls [N,H,c], u_prev [N,m] or None.  Returns device tensors X [N,c,H+1], U [N,m,H], obj [N], status [N],
    iters [N,2].
    """
    if sat is None:
        raise TypeError('sat is mandatory: the reference fails at optimize.py:43 without it')
    lib = _lib.lib()
    Xb = _lib.dev(X_bm, np.complex128)
    n, c, H1 = Xb.shape
    H = H1 - 1
    Ub = _lib.dev(np.real(U_bm) if not hasattr(U_bm, 'device') else U_bm, np.float64)
    m = Ub.shape[1]
    _lib.require_shape(c, m)
    xi = _lib.dev(x_init, np.complex128)
    Q = _lib.dev(Q_ls, np.complex128)
    R = _lib.dev(np.real(R_ls) if not hasattr(R_ls, 'device') else R_ls, np.float64)
    A = _lib.dev(A_ls, np.complex128)
    B = _lib.dev(B_ls, np.complex128)
    D = _lib.dev(Delta_ls, np.complex128)
    up = None if (u_prev is None or du is None) else _lib.dev(np.real(u_prev), np.float64)
    X = _lib.empty((n, c, H + 1), np.complex128)
    U = _lib.empty((n, m, H), np.float64)
    obj = _lib.empty((n,), np.float64)
    status = _lib.empty((n,), np.int32)
    iters = _lib.empty((n, 2), np.int32)
    st = settings if settings is not None else _lib.qp_settings(kkt_fallback=2 if H > 64 else (1 if H >= 32 else 0))
    ws_bytes = lib.m4q_qp_workspace_bytes_kkt if st.kkt_fallback else lib.m4q_qp_workspace_bytes
    ws = _lib.empty((int(ws_bytes(n, c, m, H)),), np.uint8)
    _lib.check(lib.m4q_qp_admm_batched(n, c, m, H, _lib.ptr(xi), _lib.ptr(Xb), _lib.ptr(Ub), _lib.ptr(Q), _lib.ptr(R),
                                       _lib.ptr(A), _lib.ptr(B), _lib.ptr(D), _lib.ptr(up), float(sat),
                                       float(du) if du is not None else 0.0, int(up is not None), st,
                                       _lib.ptr(X), _lib.ptr(U), _lib.ptr(obj), _lib.ptr(status), _lib.ptr(iters),
                                       _lib.ptr(ws), _lib.stream_ptr()))
    return X, U, obj, status, iters


def quad_program(x_init, X_bm, U_bm, Q_ls, R_ls, A_ls, B_ls, Delta_ls, u_prev=None, sat=None, du=None, verbose=False,
                 settings=None):
    """Same arguments and returns as optimize.py:12-60: (X [c,H+1] complex, U [m,H] real, obj_val, info)."""
    X_bm = np.atleast_2d(np.asarray(X_bm, dtype=complex))
    U_bm = np.atleast_2d(np.real(np.asarray(U_bm)))
    c = X_bm.shape[0]
    m, H = U_bm.shape
    Q = np.stack([np.asarray(q, dtype=complex) for q in Q_ls])
    R = np.stack([np.real(np.asarray(r)).reshape(m, m) for r in R_ls])
    A = np.stack([np.asarray(a, dtype=complex) for a in A_ls])
    B = np.stack([np.asarray(b, dtype=complex).reshape(c, m) for b in B_ls])
    D = np.stack([np.asarray(dl, dtype=complex).reshape(c) for dl in Delta_ls])
    up = None if u_prev is None else np.real(np.asarray(u_prev)).reshape(1, m)
    X, U, obj, status, iters = quad_program_batched(
        np.asarray(x_init, dtype=complex).reshape(1, c), X_bm[None], U_bm[None], Q[None], R[None], A[None], B[None],
        D[None], up, sat, du, settings)
    status = int(status[0])
    obj_val = float(obj[0]) if status != 3 else np.inf
    info = QPInfo(status, obj_val, *iters[0].cpu().numpy())
    if verbose:
        print('m4q qp: status %s, %d ADMM iterations, %d factorizations, objective %.6e'
              % (info.status, info.admm_iterations, info.factorizations, obj_val))
    if status == 2:
        import warnings
        warnings.warn('Solution may be inaccurate.', UserWarning)
    return X[0].cpu().numpy(), U[0].cpu().numpy(), obj_val, info
