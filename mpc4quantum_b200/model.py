"""Surrogate-model containers -- API of mpc4quantum/model.py.

``DMDc`` (model.py:7-103) is the read-only container on the MPC hot path: ``get_discrete()`` hands the blocks
``[A_x | A_u]`` to the device once, when the closed-loop plan is built.

``DiscrepDMDc`` (model.py:109-213) and ``OnlineDMDc`` (model.py:216-313) are the data-driven variants that
``mpc(streaming=True)`` updates after every MPC step (mpc.py:281-285).  They are small dense host-side updates
(one pseudo-inverse, or one rank-1 recursive-least-squares step, per MPC step) and run in numpy.

Reference behaviour kept on purpose: both ``fit_iteration`` implementations REBIND ``self.A`` to a new array.  The
controller inside ``mpc()`` linearises through operators captured before the loop (mpc.py:156, linearize.py:13-32),
so a streaming run keeps controlling with the model it started from; the updates are visible to ``model.predict``
(the steps between plant measurements, mpc.py:264-267) and in the model that ``mpc()`` returns.
"""
import numpy as np


class DMDc:
    """y = A_x x + A_u u with A = [A_x | A_u] (model.py:11-31, 81-103)."""

    def __init__(self, dim_y, dim_x, dim_u, A0):
        self.dim_y = dim_y
        self.dim_x = dim_x
        self.dim_u = dim_u
        self.A = A0
        self.discount = 1
        self.rcond = 1e-15

    @classmethod
    def from_data(cls, Y, X, U, **kwargs):
        raise NotImplementedError()

    @classmethod
    def from_bootstrap(cls, dim_y, dim_x, dim_u, A0, **kwargs):
        raise NotImplementedError()

    @classmethod
    def from_randn(cls, dim_y, dim_x, dim_u, **kwargs):
        raise NotImplementedError()

    def fit_iteration(self, next_y, next_x, next_u):
        raise NotImplementedError()

    def predict(self, current_x, current_u):
        A_x, A_u = self.get_discrete()
        return A_x @ np.reshape(current_x, (self.dim_x, -1)) + A_u @ np.reshape(current_u, (self.dim_u, -1))

    def get_discrete(self):
        return self.A[:self.dim_y, :self.dim_x], self.A[:self.dim_y, self.dim_x:]


def _regressors(X, U):
    """Z = [X; U] and dim_u for an optional control block."""
    if U is None:
        return X, 0
    return np.vstack([X, U]), U.shape[0]


class _History:
    """Optional in-memory history of the fitted operators, every `_isave` iterations (model.py:131-135, 235-239)."""

    def _init_history(self):
        self._save = False
        self._iteration = 0
        self._isave = 10

    def _tick(self):
        self._iteration += 1
        return self._save and self._iteration % self._isave == 0


class DiscrepDMDc(DMDc, _History):
    """Discrepancy DMDc (model.py:109-213): keeps (discounted) snapshot stacks and, once the state stack has rank
    `min_rank`, adds the least-squares fit of the current prediction error to the model."""

    def __init__(self, dim_y, dim_x, dim_u, A0, **kwargs):
        super().__init__(dim_y, dim_x, dim_u, A0)
        self.initialization = kwargs
        self.Y = kwargs.get('Y')
        self.X = kwargs.get('X')
        self.U = kwargs.get('U')
        self.discount = kwargs.get('discount', self.discount)
        self.rcond = kwargs.get('rcond', self.rcond)
        self.min_rank = dim_x
        self.iA = [A0]
        self._init_history()

    @classmethod
    def from_randn(cls, dim_y, dim_x, dim_u, **kwargs):
        """A0 ~ sigma * N(0, 1), real (global numpy RNG, as the reference: model.py:137-150)."""
        sigma = kwargs['sigma']
        return cls(dim_y, dim_x, dim_u, sigma * np.random.randn(dim_y, dim_x + dim_u), sigma=sigma)

    @classmethod
    def from_bootstrap(cls, dim_y, dim_x, dim_u, A0, **kwargs):
        return cls(dim_y, dim_x, dim_u, A0)

    @classmethod
    def from_data(cls, Y, X, U=None, **kwargs):
        """A0 = Y pinv([X; U], rcond) (model.py:157-178)."""
        rcond = kwargs['rcond']
        Z, dim_u = _regressors(X, U)
        return cls(Y.shape[0], X.shape[0], dim_u, Y @ np.linalg.pinv(Z, rcond=rcond), Y=Y, X=X, U=U, rcond=rcond)

    @staticmethod
    def _update_stack(val, stack, discount, nadd=1):
        cols = np.reshape(val, (-1, nadd))
        return cols if stack is None else np.hstack([discount * stack, cols])

    def fit_iteration(self, next_y, next_x, next_u=np.array([])):
        self.Y = self._update_stack(next_y, self.Y, self.discount)
        self.X = self._update_stack(next_x, self.X, self.discount)
        self.U = self._update_stack(next_u, self.U, self.discount)
        if np.linalg.matrix_rank(self.X) >= self.min_rank:
            residual = self.Y - self.predict(self.X, self.U)
            self.A = self.A + residual @ np.linalg.pinv(np.vstack([self.X, self.U]), rcond=self.rcond)
        if self._tick():
            self.iA.append(np.copy(self.A))
        return self.get_discrete()

    def append(self, Y, X, U):
        n = Y.shape[1]
        self.Y = self._update_stack(Y, self.Y, 1, n)
        self.X = self._update_stack(X, self.X, 1, n)
        self.U = self._update_stack(U, self.U, 1, n)


class OnlineDMDc(DMDc, _History):
    """Recursive-least-squares DMDc (model.py:216-313; Zhang et al., online DMD): with z = [x; u],
    gamma = 1 / (1 + z^T P z),  A += gamma (y - A z) (P z)^T,  P = (P - gamma (P z)(P z)^T) / discount.
    The products use the plain transpose, also for complex data, as the reference does (model.py:300-305)."""

    def __init__(self, dim_y, dim_x, dim_u, P0, A0, **kwargs):
        super().__init__(dim_y, dim_x, dim_u, A0)
        self.initialization = kwargs
        self.P = P0
        self.iP = [P0]
        self.iA = [A0]
        self._init_history()

    @classmethod
    def from_randn(cls, dim_y, dim_x, dim_u, **kwargs):
        dim_z = dim_x + dim_u
        P0 = kwargs['alpha'] * np.identity(dim_z)
        return cls(dim_y, dim_x, dim_u, P0, kwargs['sigma'] * np.random.randn(dim_y, dim_z), **kwargs)

    @classmethod
    def from_bootstrap(cls, dim_y, dim_x, dim_u, A0, **kwargs):
        return cls(dim_y, dim_x, dim_u, kwargs['alpha'] * np.identity(dim_x + dim_u), A0, **kwargs)

    @classmethod
    def from_data(cls, Y, X, U=None, **kwargs):
        Z, dim_u = _regressors(X, U)
        P0 = np.linalg.pinv(Z @ Z.T)
        return cls(Y.shape[0], X.shape[0], dim_u, P0, Y @ Z.T @ P0, Y=Y, X=X, U=U)

    def fit_iteration(self, next_y, next_x, next_u=np.array([])):
        y = np.reshape(next_y, (-1, 1))
        z = np.vstack([np.reshape(next_x, (-1, 1)), np.reshape(next_u, (-1, 1))])
        Pz = self.P @ z
        gamma = 1 / (1 + z.T @ Pz)
        self.A = self.A + gamma * (y - self.A @ z) @ Pz.T
        self.P = (self.P - gamma * Pz @ Pz.T) / self.discount
        if self._tick():
            self.iA.append(np.copy(self.A))
            self.iP.append(np.copy(self.P))
        return self.get_discrete()


class DMDcEnsemble:
    """N perturbed MODELS of one shape for ``mpc_ensemble``: member k controls with ``A[k]`` = [A_x | A_u] of its own
    (additive to the reference API; one ``DMDc`` per member, model.py:11-31, without N Python objects).

    ``A`` is a host array or CUDA tensor [N, dim_y, dim_x + dim_u], e.g. the output of
    ``vectorize.discretize_homogeneous_batched`` for N sets of Liouvillians.
    """

    def __init__(self, dim_y, dim_x, dim_u, A):
        self.dim_y, self.dim_x, self.dim_u = dim_y, dim_x, dim_u
        self.A = A

    def __len__(self):
        return self.A.shape[0]

    def member(self, k):
        A = self.A[k]
        return DMDc(self.dim_y, self.dim_x, self.dim_u, A.cpu().numpy() if hasattr(A, 'cpu') else np.asarray(A))

    def slice(self, lo, hi):
        return DMDcEnsemble(self.dim_y, self.dim_x, self.dim_u, self.A[lo:hi])

    def get_discrete(self):
        """Operators of member 0 (shape checks, library size)."""
        return self.member(0).get_discrete()


class ExactModel:
    """Exact-discretisation model mode (SURVEY.md section 8f rank 1; no counterpart in the reference, whose models
    are the order-k Taylor blocks of vectorize.py:8-49):  x+ = expm((L_0 + sum_i u_i L_i) dt) x.

    ``generators`` = [L_0, L_1, ..., L_m], continuous-time c x c matrices (e.g. Liouvillians from ``vectorize_me``).
    Handed to ``mpc`` / ``mpc_ensemble`` in place of a ``DMDc`` (``order`` is then ignored): the linearisation along
    the guess is A_t = expm(G(u_t) dt), B_t = the Frechet derivative of that exponential applied to x_t, Delta_t = -B_t u_t,
    evaluated on the device (``m4q_exact_linearize_batched`` stand-alone, inlined in the fused loop).
    """

    def __init__(self, generators, dt):
        self.generators = np.stack([np.asarray(g, dtype=complex) for g in generators])
        self.dt = float(dt)
        self.dim_x = self.dim_y = self.generators.shape[1]
        self.dim_u = self.generators.shape[0] - 1

    def get_model_along_traj(self, xs, us, ts=None):
        """xs [c, >= H+1], us [m, H] -> lists (A_t, B_t, Delta_t) like WrapModel.get_model_along_traj (linearize.py:61-70)."""
        from . import _lib
        us = np.atleast_2d(np.real(np.asarray(us)))
        H = us.shape[1]
        A, B, D = self._along(np.asarray(xs, dtype=complex)[None, :, :H + 1], us[None], H)
        return list(A[0].cpu().numpy()), list(B[0].cpu().numpy()), [d.reshape(-1, 1) for d in D[0].cpu().numpy()]

    def _along(self, xs, us, H):
        from . import _lib
        lib = _lib.lib()
        c, m = self.dim_x, self.dim_u
        _lib.require_shape(c, m)
        Xg = _lib.dev(xs, np.complex128)
        Ug = _lib.dev(np.real(us), np.float64)
        nb = Xg.shape[0]
        gen = _lib.dev(self.generators, np.complex128)
        A_out = _lib.empty((nb, H, c, c), np.complex128)
        B_out = _lib.empty((nb, H, c, m), np.complex128)
        D_out = _lib.empty((nb, H, c), np.complex128)
        _lib.check(lib.m4q_exact_linearize_batched(nb, c, m, H, self.dt, _lib.ptr(gen), _lib.ptr(Xg), _lib.ptr(Ug),
                                                   _lib.ptr(A_out), _lib.ptr(B_out), _lib.ptr(D_out), _lib.stream_ptr()))
        return A_out, B_out, D_out
