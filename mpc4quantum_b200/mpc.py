"""Receding-horizon driver -- API of mpc4quantum/mpc.py, with the loop itself on the device.

``mpc()`` keeps the reference signature and return convention (mpc.py:128-129, 294-304).  For the quantum plants of
this package the whole closed loop (linearise -> QP -> line search -> plant -> shift, every MPC step) runs inside one
launch of the fused sm_100a kernel behind ``m4q_mpc_closed_loop``; a user-defined ``Experiment`` or an
``exit_condition`` callback is served by stepping the same kernel one MPC step at a time with the plant on the host.
``mpc_ensemble()`` is the additive extension: N perturbed plants, one warp each.
"""
import ctypes as ct
import warnings

import numpy as np

from . import _lib
from .linearize import WrapModel, create_library, krtimes, model_blocks, size_of_library, create_power_list
from .model import DMDcEnsemble, ExactModel


class StepClock:
    """Time grid of the loop (mpc.py:14-35)."""

    def __init__(self, dt, horizon, n_steps):
        self.dt = float(dt)
        self.horizon = horizon
        self.n_steps = n_steps
        self.measure_freq = 1
        self.ts = np.arange(self.n_steps) * self.dt
        self.ts_sim = self.ts

    def set_endsim(self, index):
        self.ts_sim = self.ts[:index]

    def ts_step(self, a_step):
        return np.linspace(self.dt * (a_step + 1 - self.measure_freq), self.dt * (a_step + 1), self.measure_freq + 1)

    def ts_horizon(self, a_step):
        return self.dt * (a_step + np.arange(self.horizon))

    def to_string(self):
        pairs = [('mf', self.measure_freq), ('dt', self.dt), ('h', self.horizon), ('n', self.n_steps)]
        return '_'.join('%s_%s' % (k, val_to_str(v)) for k, v in pairs)


def val_to_str(val):
    """1.0 -> '1d0e00', 0.25 -> '2d5em01' (mpc.py:64-68)."""
    return f'{val:.1E}'.replace('E', 'e').replace('.', 'd').replace('-', 'm').replace('+', '')


def shift_guess(data):
    """Drop the first column, repeat the last (mpc.py:71-73)."""
    return np.concatenate([data[:, 1:], data[:, -1:]], axis=1)


def isinf_warning():
    warnings.warn("Solution was infinite (failed to converge). Inspect the model for accuracy, "
                  "check if control constraints can regularize the problem, "
                  "or run with verbose=True for more information.")


def real_to_complex(z):
    half = len(z) // 2
    return z[:half] + 1j * z[half:]


def complex_to_real(z):
    return np.concatenate((np.real(z), np.imag(z)))


def complex_to_real_op(P):
    P = np.asarray(P)
    return np.block([[P.real, -P.imag], [P.imag, P.real]])


def real_to_complex_op(P):
    row, col = P.shape
    return P[:row // 2, :col // 2] + 1j * P[row // 2:, :col // 2]


def iqp_line_search_batched(Q_ls, R_ls, X_htarg, U_htarg, X_guess, U_guess, X_opt, U_opt):
    """Device front end: guesses/optima carry a leading instance axis; costs and targets are shared."""
    lib = _lib.lib()
    Xg = _lib.dev(X_guess, np.complex128)
    n, c, H1 = Xg.shape
    H = H1 - 1
    Ug = _lib.dev(np.real(U_guess), np.float64)
    m = Ug.shape[1]
    Q = _lib.dev(np.stack([np.asarray(q, dtype=complex) for q in Q_ls]), np.complex128)
    R = _lib.dev(np.stack([np.real(np.asarray(r)).reshape(m, m) for r in R_ls]), np.float64)
    Xr = _lib.dev(np.atleast_2d(X_htarg), np.complex128)
    Ur = _lib.dev(np.real(np.atleast_2d(U_htarg)), np.float64)
    Xo = _lib.dev(X_opt, np.complex128)
    Uo = _lib.dev(np.real(U_opt), np.float64)
    alpha = _lib.empty((n,), np.float64)
    step = _lib.empty((n,), np.float64)
    ws = _lib.empty((int(lib.m4q_line_search_workspace_bytes(c, m, H)),), np.uint8)
    _lib.check(lib.m4q_line_search_batched(n, c, m, H, _lib.ptr(Q), _lib.ptr(R), _lib.ptr(Xr), _lib.ptr(Ur),
                                           _lib.ptr(Xg), _lib.ptr(Ug), _lib.ptr(Xo), _lib.ptr(Uo), _lib.ptr(alpha),
                                           _lib.ptr(step), _lib.ptr(ws), _lib.stream_ptr()))
    return alpha, step


def iqp_line_search(Q_ls, R_ls, X_htarg, U_htarg, X_guess, U_guess, X_opt, U_opt):
    """Exact minimiser along (opt - guess) of the reference's quadratic (mpc.py:101-125).

    Returns (alpha, new_step, new_fval, new_slope) like the reference; alpha and new_step come from the device
    kernel, which reproduces the reference's pairing of a time-major metric with state-major vectors.
    """
    alpha, step = iqp_line_search_batched(Q_ls, R_ls, X_htarg, U_htarg, np.asarray(X_guess)[None],
                                          np.asarray(U_guess)[None], np.asarray(X_opt)[None], np.asarray(U_opt)[None])
    alpha, step = float(alpha[0]), float(step[0])

    def zvec(X, U):
        return np.concatenate((complex_to_real(np.asarray(X).flatten()), complex_to_real(np.asarray(U).flatten())))
    # the two diagnostic values the reference also returns (never used by mpc()); cheap host bookkeeping
    w_blocks = [complex_to_real_op(q) for q in Q_ls] + [complex_to_real_op(r) for r in R_ls]
    Zt, Zg, Zo = zvec(X_htarg, U_htarg), zvec(X_guess, U_guess), zvec(X_opt, U_opt)
    Zn = Zg + alpha * (Zo - Zg) - Zt
    MZ = np.zeros_like(Zn)
    o = 0
    for b in w_blocks:
        k = b.shape[0]
        MZ[o:o + k] = 0.5 * (b + b.T) @ Zn[o:o + k]
        o += k
    return alpha, step, float(Zn @ MZ) / 2, MZ


# ----------------------------------------------------------------------------------------------------------
# Device plan of one closed-loop problem
# ----------------------------------------------------------------------------------------------------------
class EnsembleResult:
    """Outputs of mpc_ensemble (device tensors unless converted with .numpy())."""
    __slots__ = ('xs', 'us', 'exit_code', 'steps_done', 'qp_count', 'counters', 'fidelity', 'model_A', 'model_P')

    def __init__(self, **kw):
        for k in self.__slots__:
            setattr(self, k, kw.get(k))

    def numpy(self):
        return EnsembleResult(**{k: (getattr(self, k).cpu().numpy() if getattr(self, k) is not None else None)
                                 for k in self.__slots__})


class ClosedLoopPlan:
    """Shared problem data resident on the device + output buffers for up to `capacity` members.

    Mirrors the argument list of mpc() (mpc.py:128-129).  ``run`` launches the fused kernel on device-resident
    plant data; nothing in it synchronises with the host.
    """

    def __init__(self, dim_u, order, X_targ, U_targ, clock, model, Q, R, Qf, sat, du, d, lift_mode=_lib.LIFT_IDENTITY,
                 max_iter=100, warm_start=True, fid_target=None, exit_infidelity=0.0, settings=None, capacity=1,
                 external_plant=False):
        if sat is None:
            raise TypeError('sat is mandatory: the reference fails at optimize.py:43 without it')
        lib = _lib.lib()
        _lib.require_cuda()
        self.exact = isinstance(model, ExactModel)
        if self.exact:                                        # exact-discretisation mode: generators, no monomial library
            if model.dim_u != dim_u:
                raise ValueError('ExactModel has %d controls, dim_u = %d' % (model.dim_u, dim_u))
            if abs(model.dt - clock.dt) > 1e-15 * abs(clock.dt):
                raise ValueError('ExactModel.dt = %g differs from clock.dt = %g' % (model.dt, clock.dt))
            self.c, self.m, self.p = model.dim_x, dim_u, dim_u
            powers = np.eye(dim_u, dtype=np.int32)
        else:
            A_x, A_u = model.get_discrete()
            wrapped = WrapModel(A_x, A_u, dim_u, order)       # validates the library size (linearize.py:23-24)
            self.c, self.m, self.p = wrapped.dim_x, dim_u, wrapped.polyu_dim
            powers = wrapped.powers
        _lib.require_shape(self.c, self.m)
        self.d = int(d)
        self.H, self.S = int(clock.horizon), int(clock.n_steps)
        self.external = bool(external_plant)
        self.xdim = self.c if self.external else self.d * self.d
        X_targ = np.atleast_2d(np.asarray(X_targ, dtype=complex))
        U_targ = np.atleast_2d(np.real(np.asarray(U_targ)))
        n_targ = self.S + self.H + 1
        if X_targ.shape[1] < self.S + self.H or U_targ.shape[1] < self.S + self.H - 1:
            raise ValueError('targets must cover n_steps + horizon columns')
        Xt = np.zeros((self.c, n_targ), dtype=complex)
        k = min(n_targ, X_targ.shape[1])
        Xt[:, :k] = X_targ[:, :k]
        Xt[:, k:] = X_targ[:, k - 1:k]
        Ut = np.zeros((self.m, n_targ - 1))
        k = min(n_targ - 1, U_targ.shape[1])
        Ut[:, :k] = U_targ[:, :k]
        Ut[:, k:] = U_targ[:, k - 1:k]
        per_member = isinstance(model, DMDcEnsemble)
        if self.exact:
            blocks = _lib.dev(model.generators, np.complex128)
            self.n_models = 0
        elif per_member:
            # [N, c, c (p+1)] -> [N, p+1, c, c]: block 0 = A_x, block k = N_k of every member (linearize.py:32)
            stack = _lib.dev(model.A, np.complex128)
            blocks = stack.reshape(len(model), self.c, self.p + 1, self.c).permute(0, 2, 1, 3).contiguous()
            self.n_models = len(model)
        else:
            blocks = _lib.dev(model_blocks(A_x, A_u), np.complex128)
            self.n_models = 0
        self._keep = dict(
            blocks=blocks,
            powers=_lib.dev(powers, np.int32),
            Q=_lib.dev(np.asarray(Q, dtype=complex).reshape(self.c, self.c), np.complex128),
            Qf=_lib.dev(np.asarray(Qf, dtype=complex).reshape(self.c, self.c), np.complex128),
            R=_lib.dev(np.real(np.asarray(R)).reshape(self.m, self.m), np.float64),
            Xt=_lib.dev(Xt, np.complex128), Ut=_lib.dev(Ut, np.float64),
            fid=None if fid_target is None else _lib.dev(np.asarray(fid_target, dtype=complex).reshape(-1),
                                                         np.complex128))
        kp = self._keep
        # Default settings: long horizons get the pivoted KKT solve behind the Riccati path (include/m4q.h, kkt_fallback):
        # as the last resort from H = 32, as the first resort after one failed certification beyond H = 64 (the order-1
        # model at H = 100 leaves the fp64 range of the cost-to-go from the fourth step on)
        st = settings if settings is not None else _lib.qp_settings(
            kkt_fallback=2 if self.H > 64 else (1 if self.H >= 32 else 0))
        # external (host-stepped) plant: d = 0 tells the library that xs holds lifted model states
        self.prob = _lib.MpcProblem(
            self.c, self.m, self.p, 0 if self.external else self.d, self.H, self.S, int(clock.measure_freq),
            int(bool(warm_start)), int(max_iter), _lib.LIFT_IDENTITY if self.external else int(lift_mode),
            int(du is not None), n_targ, float(clock.dt), float(sat), float(du) if du is not None else 0.0,
            float(exit_infidelity), kp['blocks'].data_ptr(), kp['powers'].data_ptr(), kp['Q'].data_ptr(),
            kp['Qf'].data_ptr(), kp['R'].data_ptr(), kp['Xt'].data_ptr(), kp['Ut'].data_ptr(),
            kp['fid'].data_ptr() if kp['fid'] is not None else None, st, int(per_member),
            _lib.MODEL_EXACT if self.exact else _lib.MODEL_TAYLOR)
        tb = int(lib.m4q_mpc_table_bytes(ct.byref(self.prob)))
        if tb < 0:
            _lib.check(-1)
        self.tables = _lib.empty((tb,), np.uint8)
        self.capacity = 0
        self._alloc(int(capacity))

    def _alloc(self, n):
        lib = _lib.lib()
        self.capacity = n
        self.xs = _lib.empty((n, self.xdim, self.S + 1), np.complex128)
        self.us = _lib.empty((n, self.m, self.S), np.float64)
        self.exit_code = _lib.empty((n,), np.int32)
        self.steps_done = _lib.empty((n,), np.int32)
        self.qp_count = _lib.zeros((n, self.S), np.int32)
        self.counters = _lib.zeros((n, 4), np.int32)
        self.fidelity = _lib.empty((n,), np.float64) if self._keep['fid'] is not None else None
        self.state = _lib.empty((int(lib.m4q_mpc_state_bytes(ct.byref(self.prob), n)),), np.uint8)

    def fetch(self, res):
        """Device results -> host, through pinned staging buffers owned by the plan (one asynchronous copy per array on
        the current stream, one synchronisation).  The returned numpy arrays are views of those buffers: valid until the
        next ``fetch`` of this plan (``mpc_ensemble(as_numpy=True)`` copies nothing else)."""
        t = _lib.torch()
        host = getattr(self, '_host', None)
        if host is None:
            host = self._host = {}
        out = {}
        for k in EnsembleResult.__slots__:
            v = getattr(res, k)
            if v is None:
                out[k] = None
                continue
            buf = host.get(k)
            if buf is None or buf.shape[0] < v.shape[0] or buf.shape[1:] != v.shape[1:] or buf.dtype != v.dtype:
                buf = host[k] = t.empty(tuple(v.shape), dtype=v.dtype).pin_memory()
            dst = buf[:v.shape[0]]
            dst.copy_(v, non_blocking=True)
            out[k] = dst
        t.cuda.current_stream().synchronize()
        return EnsembleResult(**{k: (None if v is None else v.numpy()) for k, v in out.items()})

    def launch_info(self, n=0):
        """Launch geometry for n members (0: the widest launch)."""
        w, c, s = _lib.c_i32(), _lib.c_i32(), _lib.c_i32()
        _lib.check(_lib.lib().m4q_mpc_launch_info(ct.byref(self.prob), int(n), ct.byref(w), ct.byref(c), ct.byref(s)))
        return dict(warps_per_cta=w.value, ctas=c.value, smem_bytes=s.value)

    def herm_sigma(self):
        """The lift's index involution sigma (list of c ints), or None when the lift has none."""
        sig = (_lib.c_i32 * max(int(self.prob.c), 1))()
        r = _lib.lib().m4q_mpc_herm_sigma(ct.byref(self.prob), sig)
        if r < 0:
            _lib.check(-1)
        return list(sig[:int(self.prob.c)]) if r == 1 else None

    def factor_counts(self):
        """Riccati factorisations of the last launch: dict(herm=..., full=...), Hermitian and realified coordinates.
        Synchronises the current stream."""
        off = int(_lib.lib().m4q_mpc_factor_counts_offset(ct.byref(self.prob)))
        if off < 0:
            _lib.check(-1)
        v = self.tables[off:off + 16].cpu().numpy().view(np.uint64)
        return dict(herm=int(v[0]), full=int(v[1]))

    def run(self, x0, H0=None, H1=None, n=None, x0_shared=False, shared_hamiltonian=False, step_begin=0,
            step_end=None, stream=None, noise_sigma=0.0, noise_seed=0, member_offset=0, streaming=None,
            fidelity_sqrt=False):
        """Enqueue the closed loop for n members.  x0/H0/H1 are CUDA tensors (complex128).

        A plan owns ONE set of tables (with the atomic work counter of the launch) and ONE set of output buffers: launches
        of one plan are serialised (a launch on another stream waits for the previous one); use one plan per stream for
        concurrent launches, and read the results of a launch before the next one of the same plan overwrites them.
        Results of members that stop early (exit codes 1/2/3) are zero beyond ``steps_done``.
        streaming = (A [n, c, c (p+1)], P [n, dz, dz], discount): per-member OnlineDMDc state, updated in place."""
        n = self.capacity if n is None else int(n)
        if self.n_models and n > self.n_models:
            raise ValueError('%d members but only %d models' % (n, self.n_models))
        if n > self.capacity:
            self._alloc(n)
        if not self.external and n > 0:
            if H0 is None or H1 is None:
                raise ValueError('plant Hamiltonians H0, H1 are required')
            if H0.shape[-1] != self.d or H0.shape[-2] != self.d:
                raise ValueError('H0 is %s, the plan was built for d = %d' % (tuple(H0.shape), self.d))
            if H1.shape[-1] != self.d or H1.shape[-3] != self.m:
                raise ValueError('H1 is %s, expected [.., dim_u = %d, %d, %d] (one drive Hamiltonian per control)'
                                 % (tuple(H1.shape), self.m, self.d, self.d))
            if not shared_hamiltonian and (H0.shape[0] < n or H1.shape[0] < n):
                raise ValueError('%d members but %d / %d Hamiltonians' % (n, H0.shape[0], H1.shape[0]))
        if n > 0 and x0.shape[-1] != self.xdim:
            raise ValueError('x0 has %d entries per member, the plant state has %d' % (x0.shape[-1], self.xdim))
        if n > 0 and not x0_shared and x0.shape[0] < n:
            raise ValueError('%d members but %d initial states (pass x0_shared=True for one shared state)' % (n, x0.shape[0]))
        step_end = self.S if step_end is None else step_end
        partial = step_begin > 0 or step_end < self.S
        # one launch of a plan in flight at a time: the tables (work counter), workspaces and output buffers belong to the
        # plan, so a launch on another stream first waits for the previous one (same stream: ordered anyway)
        t = _lib.torch()
        st = stream if stream is not None else t.cuda.current_stream()
        last = getattr(self, '_last_launch', None)
        if last is not None:
            st.wait_event(last)
        if step_begin == 0:
            with t.cuda.stream(st):          # on the launch stream, not on whatever stream is current
                self.xs[:n].zero_()
                self.us[:n].zero_()
                self.qp_count[:n].zero_()
        self.prob.noise_sigma, self.prob.noise_seed = float(noise_sigma), int(noise_seed) & (2 ** 64 - 1)
        self.prob.member_offset = int(member_offset)
        self.prob.fidelity_sqrt = int(bool(fidelity_sqrt))
        if streaming is not None:
            sA, sP, disc = streaming
            self.prob.streaming, self.prob.stream_discount = 1, float(disc)
            self.prob.stream_A, self.prob.stream_P = sA.data_ptr(), sP.data_ptr()
        else:
            self.prob.streaming, self.prob.stream_A, self.prob.stream_P = 0, None, None
        _lib.check(_lib.lib().m4q_mpc_closed_loop(
            ct.byref(self.prob), n, _lib.ptr(x0), int(x0_shared), _lib.ptr(H0), _lib.ptr(H1), int(shared_hamiltonian),
            int(step_begin), int(step_end), int(self.external), _lib.ptr(self.xs), _lib.ptr(self.us),
            _lib.ptr(self.exit_code), _lib.ptr(self.steps_done), _lib.ptr(self.qp_count), _lib.ptr(self.counters),
            _lib.ptr(self.fidelity), _lib.ptr(self.state) if (partial or self.external) else _lib.c_vp(None),
            _lib.ptr(self.tables), _lib.stream_ptr(stream)))
        self._last_launch = t.cuda.Event()
        self._last_launch.record(st)
        return EnsembleResult(xs=self.xs[:n], us=self.us[:n], exit_code=self.exit_code[:n],
                              steps_done=self.steps_done[:n], qp_count=self.qp_count[:n], counters=self.counters[:n],
                              fidelity=None if self.fidelity is None else self.fidelity[:n],
                              model_A=None if streaming is None else streaming[0][:n],
                              model_P=None if streaming is None else streaming[1][:n])


def _noise_of(experiment):
    """(sigma, seed) of an experiment with set_sigma(); a missing seed is drawn from numpy's global generator."""
    sigma = float(getattr(experiment, '_sigma', 0) or 0)
    if not sigma:
        return 0.0, 0
    seed = getattr(experiment, '_noise_seed', None)
    if seed is None:
        seed = int(np.random.randint(0, 2 ** 31 - 1)) * (2 ** 31) + int(np.random.randint(0, 2 ** 31 - 1))
    return sigma, int(seed)


def mpc_ensemble(x0, dim_u, order, X_targ, U_targ, clock, experiment, model, Q, R, Qf, sat=None, du=None, max_iter=100,
                 warm_start=True, fid_target=None, exit_infidelity=0.0, settings=None, plan=None, as_numpy=True,
                 streaming=False, fidelity_convention='prob'):
    """The loop of mpc.py:128-304 for every plant of an ``EnsembleQExperiment`` (one warp per member).

    x0 is one plant state (shared) or [N, d*d].  Returns an ``EnsembleResult``: xs [N, d*d, S+1], us [N, m, S],
    exit_code [N] (reference codes), steps_done [N], qp_count [N, S], counters [N, 4], fidelity [N] if a target
    vector is given.

    streaming=True (mpc.py:281-285) with an ``OnlineDMDc`` model: every member starts from the model's (A, P) and
    runs its own rank-1 updates on the device after every step (model.py:295-313); the final operators come back as
    ``model_A [N, c, c (p+1)]`` and ``model_P``.  As in the reference the controller keeps the operators it was built
    with; the updated ones drive the model steps between measurements (``clock.measure_freq > 1``).
    fidelity_convention: 'prob' = Re<target, x> (<psi|rho|psi> for a pure target), 'sqrt' = its square root, which is
    what the reference's figures plot (qutip.fidelity, tests/test_mpc4quantum.py:590, :691).
    experiment.set_sigma(sigma, seed): measurement noise inside the fused loop (experiment.py:193-194, :212)."""
    if fidelity_convention not in ('prob', 'sqrt'):
        raise ValueError("fidelity_convention is 'prob' or 'sqrt'")
    n = len(experiment)
    if plan is None:
        plan = ClosedLoopPlan(dim_u, order, X_targ, U_targ, clock, model, Q, R, Qf, sat, du, experiment.d,
                              experiment.lift_mode, max_iter, warm_start, fid_target, exit_infidelity, settings, n)
    x0 = np.asarray(x0, dtype=complex) if not hasattr(x0, 'cpu') else x0
    if experiment.lift_mode == _lib.LIFT_PROCESS and x0.shape[-1] == experiment.d ** 4:
        # process vectors in, propagators on the device (experiment.py:371-388)
        x0 = np.asarray(x0.cpu().numpy() if hasattr(x0, 'cpu') else x0)
        x0 = np.array([experiment.proj_unitary(v) for v in x0.reshape(-1, x0.shape[-1])]).reshape(
            x0.shape[:-1] + (experiment.d ** 2,))
    shared = x0.ndim == 1
    x0d = _lib.dev(x0.reshape(1, -1) if shared else x0, np.complex128)
    H0 = _lib.dev(experiment.H0, np.complex128)
    H1 = _lib.dev(experiment.H1, np.complex128)
    stream_state = None
    if streaming:
        if not (hasattr(model, 'P') and hasattr(model, 'A')) or plan.exact:
            raise NotImplementedError('streaming inside the fused ensemble loop needs an OnlineDMDc model (A, P); '
                                      'DiscrepDMDc runs through mpc(streaming=True) on the host-stepped path')
        t = _lib.torch()
        A0 = _lib.dev(np.asarray(model.A, dtype=complex), np.complex128)
        P0 = _lib.dev(np.asarray(model.P, dtype=complex), np.complex128)
        stream_state = (A0.unsqueeze(0).repeat(n, 1, 1).contiguous(), P0.unsqueeze(0).repeat(n, 1, 1).contiguous(),
                        float(getattr(model, 'discount', 1)))
    sigma, seed = _noise_of(experiment)
    res = plan.run(x0d, H0, H1, n=n, x0_shared=shared, noise_sigma=sigma, noise_seed=seed,
                   member_offset=getattr(experiment, 'member_offset', 0), streaming=stream_state,
                   fidelity_sqrt=fidelity_convention == 'sqrt')
    return plan.fetch(res) if as_numpy else res


# ----------------------------------------------------------------------------------------------------------
# mpc(): the reference entry point
# ----------------------------------------------------------------------------------------------------------
def _device_plant(experiment):
    from .experiment import QExperiment, QProcess, QSynthesis
    if isinstance(experiment, QProcess):
        return type(experiment).simulate is QSynthesis.simulate
    return isinstance(experiment, QExperiment) and type(experiment).simulate is QExperiment.simulate


def mpc(x0, dim_u, order, X_targ, U_targ, clock, experiment, model, Q, R, Qf, sat=None, du=None, max_iter=100,
        exit_condition=None, streaming=False, warm_start=True, progress_bar=True, verbose=False):
    """Same arguments and returns as the reference (mpc.py:128-129): ([xs, us], model, exit_code).

    exit codes: 0 normal, 1 exit_condition met, 2 QP not certified, 3 non-finite QP (mpc.py:131, :195, :202, :291).
    """
    if sat is None:
        raise TypeError('sat is mandatory: the reference fails at optimize.py:43 without it')
    x0 = np.asarray(x0, dtype=complex).reshape(-1)
    fused_stream = streaming and hasattr(model, 'P') and not isinstance(model, ExactModel)     # OnlineDMDc
    if _device_plant(experiment) and exit_condition is None and (not streaming or fused_stream):
        return _mpc_fused(x0, dim_u, order, X_targ, U_targ, clock, experiment, model, Q, R, Qf, sat, du, max_iter,
                          warm_start, streaming)
    return _mpc_host_stepped(x0, dim_u, order, X_targ, U_targ, clock, experiment, model, Q, R, Qf, sat, du, max_iter,
                             exit_condition, warm_start, streaming)


def _finish(xs, us, steps_done, exit_code, clock, model):
    """Return convention of mpc.py:294-304.  xs [dim, S+1], us [m, S]; steps_done = completed MPC steps.

    An early exit "ignores the last attempted entry": the reference slices with the loop index of the step it broke
    out of, which for exit code 1 is a completed step.
    """
    if exit_code == 0:
        clock.set_endsim(steps_done)
        return [xs[:, :steps_done + 1], us[:, :steps_done]], model, exit_code
    if exit_code == 3:
        isinf_warning()
    idx = steps_done - 1 if exit_code == 1 else steps_done
    clock.set_endsim(idx)
    return [xs[:, :idx + 1], us[:, :idx] if idx > 0 else None], model, exit_code


def _mpc_fused(x0, dim_u, order, X_targ, U_targ, clock, experiment, model, Q, R, Qf, sat, du, max_iter, warm_start,
               streaming=False):
    d = experiment.H0.shape[0]
    if len(experiment.H1_list) != dim_u:
        raise IndexError('dim_u = %d but the experiment has %d drive Hamiltonians' % (dim_u, len(experiment.H1_list)))
    if x0.shape[0] != (d ** 4 if experiment.lift_mode == _lib.LIFT_PROCESS else d * d):
        raise ValueError('x0 has %d entries, the plant state has %d' % (x0.shape[0], d * d))
    plan = ClosedLoopPlan(dim_u, order, X_targ, U_targ, clock, model, Q, R, Qf, sat, du, d, experiment.lift_mode,
                          max_iter, warm_start, capacity=1)
    H0 = _lib.dev(experiment.H0[None], np.complex128)
    H1 = _lib.dev(np.stack(experiment.H1_list)[None], np.complex128)
    process = experiment.lift_mode == _lib.LIFT_PROCESS
    if process:     # the kernel carries the propagator; mpc() speaks process vectors (experiment.py:371-401)
        x0 = np.asarray(experiment.to_unitary(x0), dtype=complex)
    stream_state = None
    if streaming:
        stream_state = (_lib.dev(np.asarray(model.A, dtype=complex)[None], np.complex128),
                        _lib.dev(np.asarray(model.P, dtype=complex)[None], np.complex128), float(model.discount))
    sigma, seed = _noise_of(experiment)
    res = plan.run(_lib.dev(x0[None], np.complex128), H0, H1, n=1, noise_sigma=sigma, noise_seed=seed,
                   streaming=stream_state).numpy()
    if streaming:       # fit_iteration rebinds the operators (model.py:305-306); so does this
        model.A, model.P = res.model_A[0], res.model_P[0]
        model._iteration += int(res.steps_done[0])
    xs = res.xs[0]
    if process:
        xs = np.array([experiment.from_unitary(col) for col in xs.T]).T
    return _finish(xs, res.us[0], int(res.steps_done[0]), int(res.exit_code[0]), clock, model)


def _mpc_host_stepped(x0, dim_u, order, X_targ, U_targ, clock, experiment, model, Q, R, Qf, sat, du, max_iter,
                      exit_condition, warm_start, streaming=False):
    """User-defined plant / exit condition / streaming model: the iterative QP of each step runs on the device (one
    launch per MPC step, guesses and ADMM state stay resident), the plant, the callbacks and the model update run on
    the host (mpc.py:247-292).

    streaming (mpc.py:281-285): ``model.fit_iteration`` is called after every step with the lifted transition.  As in
    the reference, the controller keeps linearising the operators it captured before the loop (mpc.py:156 wraps
    views that ``fit_iteration`` never writes through: it rebinds ``model.A``), so the device blocks are NOT
    re-uploaded; the updated model acts through ``model.predict`` and is returned to the caller."""
    from scipy.interpolate import interp1d
    if isinstance(model, ExactModel):
        if streaming or clock.measure_freq != 1:
            raise NotImplementedError('ExactModel: streaming updates and model steps between measurements are not built')
        c, wrapped = model.dim_x, None
    else:
        c = model.get_discrete()[0].shape[1]
        wrapped = WrapModel(*model.get_discrete(), dim_u, order)
    plan = ClosedLoopPlan(dim_u, order, X_targ, U_targ, clock, model, Q, R, Qf, sat, du, d=0, max_iter=max_iter,
                          warm_start=warm_start, capacity=1, external_plant=True)
    S, mf = clock.n_steps, clock.measure_freq
    xs = [None] * (S + 1)
    us = [None] * S
    xs[0] = x0
    lifted0 = _lib.dev(np.asarray(experiment.lift(x0), dtype=complex).reshape(1, c), np.complex128)
    exit_code, step = 0, 0
    for step in range(S):
        lifted = np.asarray(experiment.lift(xs[step]), dtype=complex).reshape(-1)
        plan.xs[0, :, step] = _lib.dev(lifted, np.complex128)
        res = plan.run(lifted0, n=1, step_begin=step, step_end=step + 1)
        exit_code = int(res.exit_code[0])
        if exit_code:
            break
        us[step] = res.us[0, :, step].cpu().numpy()
        if (step + 1) % mf == 0:
            ts_step = clock.ts_step(step)
            us_step = np.vstack([us[step - j] for j in range(mf)] + [us[step]]).T
            u_fns = interp1d(ts_step, us_step, fill_value='extrapolate', kind='previous')
            xs[step + 1] = np.asarray(experiment.simulate(xs[step + 1 - mf], ts_step, u_fns))[:, -1]
        else:
            lift_u = wrapped.lift_u(us[step].reshape(-1, 1))
            lift_x = np.asarray(experiment.lift(xs[step])).reshape(-1, 1)
            xs[step + 1] = np.asarray(experiment.proj(model.predict(lift_x, krtimes(lift_u, lift_x)))).flatten()
        if streaming:
            lift_ustep = wrapped.lift_u(us[step].reshape(-1, 1))
            lift_xstep = np.asarray(experiment.lift(xs[step])).reshape(-1, 1)
            model.fit_iteration(np.asarray(experiment.lift(xs[step + 1])).reshape(-1, 1), lift_xstep,
                                krtimes(lift_ustep, lift_xstep))
        if exit_condition is not None and exit_condition(xs[step + 1], xs[step], us[step]):
            exit_code = 1
            step += 1
            break
    else:
        step = S
    done = step
    xs_arr = np.vstack([np.asarray(x, dtype=complex) for x in xs[:done + 1]]).T
    us_arr = np.vstack(us[:done]).T if done > 0 else np.zeros((dim_u, 0))
    pad_x = np.zeros((xs_arr.shape[0], S + 1), dtype=complex)
    pad_x[:, :done + 1] = xs_arr
    pad_u = np.zeros((dim_u, S))
    pad_u[:, :done] = us_arr
    return _finish(pad_x, pad_u, done, exit_code, clock, model)
