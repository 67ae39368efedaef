"""Plants ("experiments") -- API of mpc4quantum/experiment.py for the quantum classes on the MPC hot path.

The reference integrates the von Neumann equation with qutip.mesolve under a piecewise-constant control
(experiment.py:202-212, mpc.py:256-260).  Here each constant segment is the exact map rho <- U rho U^dagger with
U = expm(-i (H0 + sum_k u_k H1_k) dt), evaluated by the sm_100a kernel behind ``m4q_expm_step_batched``.
"""
from abc import ABC, abstractmethod
import math

import numpy as np

from . import _lib


def _as_matrix(op):
    return np.asarray(op.full() if hasattr(op, 'full') else op, dtype=complex)


def isqrt(n):
    """Integer square root (experiment.py:318-333)."""
    if n < 0:
        raise ValueError("Square root not defined for negative numbers.")
    return math.isqrt(n)


def split_blocks(bmatrix, nrows, ncols):
    """Sub-blocks of a block matrix, row-major over blocks (experiment.py:309-315)."""
    r, h = bmatrix.shape
    return bmatrix.reshape(r // nrows, nrows, h // ncols, ncols).swapaxes(1, 2).reshape(-1, nrows, ncols)


class Experiment(ABC):
    """Interface of a controlled plant (experiment.py:8-49): f, lift, proj, simulate."""
    lift_mode = _lib.LIFT_IDENTITY

    def __init__(self):
        self.ts = None
        self.us = None
        self.xs = None

    @abstractmethod
    def f(self, t, x, u):
        """Time derivative of the state."""

    @staticmethod
    def lift(x):
        return x

    @staticmethod
    def proj(z):
        return z

    @abstractmethod
    def simulate(self, x0, ts, us):
        """States at all times in ts, shape [dim, len(ts)], for a control function of time or an array [m, len(ts)]."""


def _controls_on_grid(us, ts):
    """Control per segment [n_seg, m]: us(ts[i]) for a callable, column i of an array otherwise.

    The plant holds the control constant over a segment (zero-order hold), which is exactly what ``mpc()`` hands over:
    an ``interp1d(..., kind='previous')`` (mpc.py:258).  The reference integrates whatever interpolant it is given
    (qutip splines an ndarray); an interp1d of any other kind is refused instead of being silently sampled as a
    zero-order hold.  Any other callable, and an array, are sampled at the left end of every segment."""
    n_seg = len(ts) - 1
    kind = getattr(us, '_kind', None)
    if kind is not None and kind != 'previous':
        raise NotImplementedError("the device plant holds the control constant over a segment: pass "
                                  "interp1d(kind='previous') (mpc.py:258), got kind=%r" % (kind,))
    if callable(us):
        cols = [np.real(np.asarray(us(ts[i]))).reshape(-1) for i in range(n_seg)]
        return np.array(cols, dtype=float).reshape(n_seg, -1)
    arr = np.atleast_2d(np.real(np.asarray(us)))
    return np.ascontiguousarray(arr[:, :n_seg].T, dtype=float)


def expm_segments(x0, H0, H1, u_seg, dt, shared=False, return_propagators=False):
    """Batched plant propagation on the device.

    x0 [N, d*d] complex, H0 [N, d, d] (or [d, d] with shared=True), H1 [N, m, d, d] (or [m, d, d]),
    u_seg [N, n_seg, m] real -> device tensor [N, n_seg, d*d] of states after each segment (+ propagators).
    """
    lib = _lib.lib()
    rho = _lib.dev(x0, np.complex128)
    n, dd = rho.shape
    d = isqrt(dd)
    u = _lib.dev(u_seg, np.float64)
    n_seg, m = u.shape[1], u.shape[2]
    H0d = _lib.dev(H0, np.complex128)
    H1d = _lib.dev(H1, np.complex128)
    if d * d != dd or H0d.shape[-1] != d or H0d.shape[-2] != d:
        raise ValueError('x0 has %d entries per member, H0 is %s: the plant state is vec(rho) of a d x d matrix'
                         % (dd, tuple(H0d.shape)))
    if H1d.shape[-3] != m or H1d.shape[-1] != d:
        raise IndexError('u_seg has %d controls per segment, H1 is %s (one drive Hamiltonian per control)'
                         % (m, tuple(H1d.shape)))
    if u.shape[0] != n or (not shared and (H0d.shape[0] != n or H1d.shape[0] != n)):
        raise ValueError('batch sizes differ: x0 %d, u_seg %d, H0 %s, H1 %s' % (n, u.shape[0], tuple(H0d.shape), tuple(H1d.shape)))
    out = _lib.empty((n, n_seg, dd), np.complex128)
    props = _lib.empty((n, n_seg, d, d), np.complex128) if return_propagators else None
    _lib.check(lib.m4q_expm_step_batched(n, d, m, n_seg, float(dt), _lib.ptr(H0d), _lib.ptr(H1d), int(shared),
                                         _lib.ptr(u), _lib.ptr(rho), _lib.ptr(out), _lib.ptr(props),
                                         _lib.stream_ptr()))
    return (out, props) if return_propagators else out


class QExperiment(Experiment):
    """Closed quantum system with Hamiltonian H0 + sum_k u_k(t) H1_k (experiment.py:175-212)."""

    def __init__(self, H0, H1_list):
        super().__init__()
        self.H0 = _as_matrix(H0)
        self.H1_list = [_as_matrix(h) for h in H1_list]
        self._me_args = {}
        self._sigma = 0

    def f(self, t, x, u):
        return self.H0 * x + np.sum([H1 * x * u1 for H1, u1 in zip(self.H1_list, u)], axis=0)

    def set_sigma(self, sigma, seed=None):
        """Measurement noise (experiment.py:193-194): sigma (N(0,1) + i N(0,1)) on every returned state.  Inside the
        fused loop the noise comes from a counter-based generator keyed by `seed` (drawn from numpy's global generator
        at call time when None, so that ``np.random.seed`` governs reproducibility as it does in the reference)."""
        self._sigma = sigma
        self._noise_seed = seed

    _DEVICE_KEYS = ('rho0', 'tlist', 'H')      # what simulate() itself sets in the reference (experiment.py:203-208)

    def set(self, key, value):
        """Keyword for qutip's mesolve in the reference (experiment.py:196-200).  The device plant is the closed-system
        propagator of H0 + sum u_k H1_k: collapse operators, expectation operators, solver options or extra arguments
        cannot be honoured and are refused instead of being ignored."""
        if key not in self._DEVICE_KEYS:
            raise NotImplementedError("QExperiment.set(%r, ...): the device plant integrates the closed system only "
                                      "(no c_ops / e_ops / options / args)" % (key,))
        self._me_args[key] = value

    def simulate(self, x0, ts, us):
        ts = np.asarray(ts, dtype=float)
        self.ts = ts
        u_seg = _controls_on_grid(us, ts)
        self.us = us
        x = np.asarray(x0, dtype=complex).reshape(1, -1)
        steps = np.diff(ts)
        cols = [x[0]]
        if len(steps) and np.allclose(steps, steps[0], rtol=1e-12, atol=0):
            out = expm_segments(x, self.H0, np.stack(self.H1_list), u_seg[None], steps[0], shared=True)
            cols += list(out[0].cpu().numpy())
        else:
            for i, h in enumerate(steps):
                x = expm_segments(x, self.H0, np.stack(self.H1_list), u_seg[None, i:i + 1], h,
                                  shared=True)[:, 0].cpu().numpy()
                cols.append(x[0])
        self.xs = np.array(cols).T
        if self._sigma:
            noise = np.random.randn(*self.xs.shape) + 1j * np.random.randn(*self.xs.shape)   # experiment.py:212
            return self.xs + noise * self._sigma
        return self.xs


class QExperiment32(QExperiment):
    """Qutrit plant observed in its qubit block (experiment.py:215-235)."""
    lift_mode = _lib.LIFT_TRUNC32

    @staticmethod
    def lift(rho33_vec):
        blk = np.asarray(rho33_vec, dtype=complex).reshape(3, 3)[:2, :2]
        return (blk / np.linalg.svd(blk, compute_uv=False).sum()).flatten()    # Qobj.unit(): trace norm

    @staticmethod
    def proj(rho22_vec):
        return np.asarray(rho22_vec).flatten()     # as the reference returns it (experiment.py:232-235)


class QCoupledExperiment(QExperiment):
    """Two identical subsystems observed through their reduced states (experiment.py:238-306)."""
    lift_mode = _lib.LIFT_COUPLED

    @staticmethod
    def lift(rhoAB_vec):
        dAB = isqrt(len(rhoAB_vec))
        dA = isqrt(dAB)
        r = np.asarray(rhoAB_vec, dtype=complex).reshape(dA, dA, dA, dA)
        return np.hstack([np.trace(r, axis1=1, axis2=3).flatten(), np.trace(r, axis1=0, axis2=2).flatten()])

    @staticmethod
    def proj(rhoA_rhoB_vec):
        half = len(rhoA_rhoB_vec) // 2
        dA = isqrt(half)
        v = np.asarray(rhoA_rhoB_vec, dtype=complex)
        return np.kron(v[:half].reshape(dA, dA), v[half:].reshape(dA, dA)).flatten()


class QSynthesis(Experiment):
    """Gate synthesis (experiment.py:336-417): the plant state is a propagator U, observed through its process
    matrix P = U (x) U^* (the "density matrix of a unitary").  ``simulate`` takes and returns process vectors.

    The reference evaluates qutip.propagator under the piecewise-constant control; here every constant segment is
    the exact factor expm(-i (H0 + sum_k u_k H1_k) dt) from ``m4q_expm_step_batched``.
    """

    def __init__(self, H0, H1_list):
        super().__init__()
        self.H0 = _as_matrix(H0)
        self.H1_list = [_as_matrix(h) for h in H1_list]
        self._prop_args = {}

    def f(self, t, x, u):
        return self.H0 * x + np.sum([H1 * x * u1 for H1, u1 in zip(self.H1_list, u)], axis=0)

    def set(self, key, value):
        """Keyword for qutip's propagator in the reference (experiment.py:351-355); only what ``simulate`` itself sets
        is accepted -- see ``QExperiment.set``."""
        if key not in ('H', 't'):
            raise NotImplementedError("QSynthesis.set(%r, ...): the device plant is the closed-system propagator" % (key,))
        self._prop_args[key] = value

    @staticmethod
    def lift(U):
        """Flat propagator (n^2,) -> flat process matrix (n^4,), P = U (x) U^* (experiment.py:357-369)."""
        n = isqrt(np.shape(U)[0])
        U = np.asarray(U, dtype=complex).reshape(n, n)
        return np.kron(U, U.conj()).flatten()

    @staticmethod
    def proj(P):
        """Flat process matrix (n^4,) -> a flat propagator equal to U up to a global phase (experiment.py:371-388):
        the first non-zero n x n block of P, block (i, j), is U[i, j] conj(U); its own (i, j) entry is |U[i, j]|^2,
        so conj(block) / sqrt(that entry) = exp(-i arg U[i, j]) U."""
        P = np.asarray(P, dtype=complex)
        n = isqrt(isqrt(P.shape[0]))
        blocks = split_blocks(P.reshape(n ** 2, n ** 2), n, n)
        U = np.zeros((n, n))
        for i, b in enumerate(blocks):
            if np.any(b):
                U = b.conj() / np.lib.scimath.sqrt(b.flatten()[i])
                break
        return U.flatten()

    def propagators(self, ts, us):
        """Segment factors V_i = expm(-i H(u_i) (ts[i+1] - ts[i])), shape [len(ts) - 1, n, n]."""
        ts = np.asarray(ts, dtype=float)
        u_seg = _controls_on_grid(us, ts)
        steps = np.diff(ts)
        n = self.H0.shape[0]
        eye = np.eye(n, dtype=complex).reshape(1, -1)
        H1 = np.stack(self.H1_list)
        if len(steps) and np.allclose(steps, steps[0], rtol=1e-12, atol=0):
            _, props = expm_segments(eye, self.H0, H1, u_seg[None], steps[0], shared=True, return_propagators=True)
            return props[0].cpu().numpy()
        out = [expm_segments(eye, self.H0, H1, u_seg[None, i:i + 1], h, shared=True,
                             return_propagators=True)[1][0, 0].cpu().numpy() for i, h in enumerate(steps)]
        return np.array(out).reshape(-1, n, n)

    def simulate(self, x0, ts, us):
        n = self.H0.shape[0]
        self.ts, self.us = ts, us
        U = QSynthesis.proj(np.asarray(x0, dtype=complex).reshape(-1)).reshape(n, n)
        cols = [QSynthesis.lift(U.flatten())]
        for V in self.propagators(ts, us):
            U = V @ U
            cols.append(QSynthesis.lift(U.flatten()))
        self.xs = np.array(cols).T
        return self.xs


class QProcess(QSynthesis):
    """``QSynthesis`` wired the way the reference's gate test means to use it (tests/test_mpc4quantum.py:48-97):
    ``mpc()`` is handed process vectors (x0 = vec(U0 (x) U0^*), dim_x = n^4 model), so the observable maps seen by
    the loop are the identity; the propagator <-> process conversions stay available as ``from_unitary`` /
    ``to_unitary``.  (With ``QSynthesis.lift`` itself the reference loop lifts the 16-vector to 256 entries at
    mpc.py:135 and stops on a shape error.)"""
    lift_mode = _lib.LIFT_PROCESS
    from_unitary = staticmethod(QSynthesis.lift)
    to_unitary = staticmethod(QSynthesis.proj)

    @staticmethod
    def lift(x):
        return x

    @staticmethod
    def proj(z):
        return z


_KINDS = {'identity': (_lib.LIFT_IDENTITY, QExperiment), 'coupled': (_lib.LIFT_COUPLED, QCoupledExperiment),
          'trunc32': (_lib.LIFT_TRUNC32, QExperiment32), 'process': (_lib.LIFT_PROCESS, QProcess)}


class EnsembleQExperiment:
    """N perturbed plants: H0 [N, d, d], H1 [N, m, d, d] complex (host arrays or CUDA tensors).

    kind = 'process' (gate synthesis): the plant state handed to and returned by ``mpc_ensemble`` is the flat
    propagator U [d*d]; the model state is vec(U (x) U^*)."""

    def __init__(self, H0, H1, kind='identity'):
        self.H0 = H0
        self.H1 = H1
        self.kind = kind
        self._sigma, self._noise_seed = 0.0, None
        self.lift_mode, self._cls = _KINDS[kind]
        self.lift = self._cls.lift
        self.proj = self._cls.proj
        if kind == 'process':     # propagator <-> process vector (the loop-facing maps above are the identity)
            self.lift_unitary = QSynthesis.lift
            self.proj_unitary = QSynthesis.proj

    def __len__(self):
        return self.H0.shape[0]

    @property
    def d(self):
        return self.H0.shape[-1]

    @property
    def dim_u(self):
        return self.H1.shape[1]

    def member(self, k):
        """The k-th plant as a single QExperiment of the matching class."""
        H0 = self.H0[k].cpu().numpy() if hasattr(self.H0, 'cpu') else self.H0[k]
        H1 = self.H1[k].cpu().numpy() if hasattr(self.H1, 'cpu') else self.H1[k]
        return self._cls(np.array(H0), [np.array(h) for h in H1])

    def slice(self, lo, hi):
        out = EnsembleQExperiment(self.H0[lo:hi], self.H1[lo:hi], self.kind)
        out._sigma, out._noise_seed = self._sigma, self._noise_seed
        out.member_offset = getattr(self, 'member_offset', 0) + lo
        return out

    def set_sigma(self, sigma, seed=None):
        """Measurement noise of every member (``QExperiment.set_sigma``); the stream of member k depends on
        (seed, global index of k, MPC step, component) only.  Process ensembles (gate synthesis) refuse it: their
        plant state is a propagator, and the reference defines no measurement noise for one (QSynthesis has no
        set_sigma)."""
        if self.kind == 'process' and sigma:
            raise NotImplementedError('measurement noise is not defined for process (gate-synthesis) ensembles')
        self._sigma, self._noise_seed = float(sigma), seed

    def simulate(self, x0, u_seg, dt, return_propagators=False):
        """x0 [N, d*d], u_seg [N, n_seg, m] -> device tensor [N, n_seg, d*d]."""
        return expm_segments(x0, self.H0, self.H1, u_seg, dt, shared=False, return_propagators=return_propagators)
