"""Local linearisation of the discrete bilinear-polynomial model -- API of mpc4quantum/linearize.py.

The arithmetic of ``WrapModel`` (linearize.py:37-77) runs in the sm_100a kernel behind
``m4q_linearize_batched``; the monomial-table helpers (linearize.py:92-164) are host-side index bookkeeping
and stay in Python.
"""

import numpy as np

from . import _lib


# ----------------------------------------------------------------------------------------------------------
# Monomial tables (linearize.py:92-164)
# ----------------------------------------------------------------------------------------------------------
def multinomial_powers(n, k):
    """Exponent tuples of the expansion (x_1 + ... + x_k)^n, in the reference's order (linearize.py:92-110).

    Generated as compositions of n into k non-negative parts in ascending lexicographic order.
    """
    def compositions(total, parts):
        if parts == 1:
            yield (total,)
            return
        for first in range(total + 1):
            for rest in compositions(total - first, parts - 1):
                yield (first,) + rest
    for comp in compositions(n, k):
        yield np.array(comp, dtype=int)


def create_power_list(order, dimension):
    """All exponent tuples of total degree <= order; row 0 is the constant (linearize.py:113-116)."""
    return [pw[:-1][::-1] for pw in multinomial_powers(order, dimension + 1)]


def size_of_library(order, dimension):
    return len(create_power_list(order, dimension))


def _monomial(x, powers):
    out = np.ones_like(np.asarray(x)[0, :], dtype=np.result_type(x, float))
    for i, e in enumerate(powers):
        out = out * (np.zeros_like(out) if e < 0 else np.power(x[i, :], e))
    return out


def create_library_from_list(power_list):
    """Callables x [dim, n] -> prod_i x_i**p_i; a negative exponent gives 0 (linearize.py:123-128)."""
    return [lambda x, ps=tuple(int(e) for e in powers): _monomial(x, ps) for powers in np.array(power_list)]


def create_library(order, dimension):
    return create_library_from_list(create_power_list(order, dimension))


def diff_library(order, dimension):
    """Derivative library: (functions per control, coefficients per control)  (linearize.py:131-164)."""
    plist = np.vstack(create_power_list(order, dimension)[1:])
    fns, coefs = [], []
    for i in range(dimension):
        lowered = plist.copy()
        lowered[:, i] -= 1
        fns.append(create_library_from_list(lowered))
        coefs.append(plist[:, [i]])
    return fns, coefs


def krtimes(A, B):
    """Column-wise Kronecker (Khatri-Rao) product (linearize.py:80-89)."""
    A = np.asarray(A)
    B = np.asarray(B)
    if A.shape[1] != B.shape[1]:
        raise ValueError("Cols of A =/ Cols of B")
    return (A[:, None, :] * B[None, :, :]).reshape(A.shape[0] * B.shape[0], -1)


def model_blocks(A_op, N_op):
    """[A | N_1 | ... | N_p] -> array [p+1, c, c] (linearize.py:32: N_op.reshape(c, p, c))."""
    A_op = np.asarray(A_op, dtype=complex)
    N_op = np.asarray(N_op, dtype=complex)
    c = A_op.shape[1]
    p = N_op.shape[1] // c
    return np.concatenate([A_op[None, :c, :], N_op.reshape(c, p, c).transpose(1, 0, 2)], axis=0)


# ----------------------------------------------------------------------------------------------------------
# WrapModel
# ----------------------------------------------------------------------------------------------------------
class WrapModel:
    """x+ = A x + N (phi(u) (x) x) and its Jacobians (linearize.py:8-77), evaluated on the device."""

    def __init__(self, A_op, N_op, dim_u, order):
        self.A = A_op
        self.N = N_op
        self.dim_x = self.A.shape[1]
        self.dim_u = dim_u
        self.order = order
        self.polyu_dim = int(self.N.shape[1] / self.dim_x)
        if size_of_library(self.order, self.dim_u) - 1 != self.polyu_dim:
            raise ValueError("Dimension mismatch when wrapping a model operator.")
        self.powers = np.vstack(create_power_list(order, dim_u)[1:]).astype(np.int32)
        self.fns = create_library(self.order, self.dim_u)[1:]
        self.deriv_fns, self.deriv_coefs = diff_library(self.order, self.dim_u)
        self.unpacked_N = np.asarray(N_op).reshape(self.dim_x, self.polyu_dim, self.dim_x)

    def lift_u(self, u_shaped):
        return np.vstack([f(u_shaped) for f in self.fns])

    # -- device evaluation -------------------------------------------------------------------------------
    def _along(self, xs, us, H):
        """Batched front end: xs [B, c, H+1] complex, us [B, m, H] -> A [B,H,c,c], B [B,H,c,m], D [B,H,c]."""
        lib = _lib.lib()
        c, m, p = self.dim_x, self.dim_u, self.polyu_dim
        _lib.require_shape(c, m)
        Xg = _lib.dev(xs, np.complex128)
        Ug = _lib.dev(np.real(us), np.float64)
        nb = Xg.shape[0]
        blocks = _lib.dev(model_blocks(self.A, self.N), np.complex128)
        powers = _lib.dev(self.powers, np.int32)
        A_out = _lib.empty((nb, H, c, c), np.complex128)
        B_out = _lib.empty((nb, H, c, m), np.complex128)
        D_out = _lib.empty((nb, H, c), np.complex128)
        _lib.check(lib.m4q_linearize_batched(nb, c, m, p, H, _lib.ptr(blocks), _lib.ptr(powers), _lib.ptr(Xg),
                                             _lib.ptr(Ug), _lib.ptr(A_out), _lib.ptr(B_out), _lib.ptr(D_out),
                                             _lib.stream_ptr()))
        return A_out, B_out, D_out

    def _point(self, x, u):
        x = np.asarray(x, dtype=complex).reshape(-1)
        u = np.real(np.asarray(u)).reshape(-1)
        xs = np.stack([x, x], axis=1)[None]
        A, B, D = self._along(xs, u.reshape(1, -1, 1), 1)
        return A[0, 0].cpu().numpy(), B[0, 0].cpu().numpy(), D[0, 0].cpu().numpy()

    def f(self, x, u, t):
        A, B, D = self._point(x, u)
        xv = np.asarray(x, dtype=complex).reshape(-1)
        uv = np.real(np.asarray(u)).reshape(-1)
        return (A @ xv + B @ uv + D).reshape(-1, 1)

    def df_dx(self, x, u, t):
        return self._point(x, u)[0]

    def df_du(self, x, u, t):
        return self._point(x, u)[1]

    def get_model_along_traj(self, xs, us, ts):
        H = len(ts)
        xs = np.asarray(xs, dtype=complex)
        us = np.real(np.asarray(us))
        if xs.shape[1] < H + 1:   # the reference only reads the first len(ts) columns
            xs = np.hstack([xs, xs[:, -1:]])
        A, B, D = self._along(xs[None, :, :H + 1], us[None, :, :H], H)
        A, B, D = A[0].cpu().numpy(), B[0].cpu().numpy(), D[0].cpu().numpy()
        return [A[i] for i in range(H)], [B[i] for i in range(H)], [D[i].reshape(-1, 1) for i in range(H)]

    def get_model_from_initial(self, xs, us, ts):
        A, B, D = self._point(xs[:, 0], us[:, 0])
        return [A] * len(ts), [B] * len(ts), [D.reshape(-1, 1)] * len(ts)
