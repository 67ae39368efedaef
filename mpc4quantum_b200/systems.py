"""Benchmark systems and ensemble draws, stated with plain numpy (no qutip).

Specification source: the reference's test utilities and state-preparation tests
(/root/reference/tests/util_qubits.py:19-138, tests/test_mpc4quantum.py:281-368, 504-564, 607-670)
and the ensemble definitions of SURVEY.md section 8(d).  These are *inputs*: host-side, built once.
"""
import numpy as np

from .experiment import QExperiment, QCoupledExperiment, QExperiment32, EnsembleQExperiment
from .model import DMDc
from .mpc import StepClock
from .vectorize import discretize_homogeneous, liouvillian

SX = np.array([[0, 1], [1, 0]], dtype=complex)
SY = np.array([[0, -1j], [1j, 0]], dtype=complex)
SZ = np.array([[1, 0], [0, -1]], dtype=complex)
I2 = np.eye(2, dtype=complex)


def rx(phi):
    """Single-qubit x rotation exp(-i phi sx / 2) (qutip.qip.operations.rx)."""
    c, s = np.cos(phi / 2), np.sin(phi / 2)
    return np.array([[c, -1j * s], [-1j * s, c]], dtype=complex)


def proj(d, k):
    out = np.zeros((d, d), dtype=complex)
    out[k, k] = 1
    return out


def destroy(d):
    return np.diag(np.sqrt(np.arange(1, d)), 1).astype(complex)


class RWA_Qubit:
    """tests/util_qubits.py:60-80: H0 = (wQ - wR)/2 sz, H1 = sx/2."""

    def __init__(self, wQ, wD, wR):
        self.dim_s, self.dim_x, self.dim_u = 2, 4, 1
        self._w0, self._wD, self._wR = wQ, wD, wR
        H0 = 0.5 * (wQ - wR) * SZ
        H1 = 0.5 * SX
        self.H_list = [H0, H1]
        self.QE = QExperiment(H0, [H1])


class RWA_Transmon:
    """tests/util_qubits.py:92-111: H0 = alpha |2><2|, HX = (a^+ + a)/2, HY = i (a^+ - a)/2."""
    _QE = QExperiment

    def __init__(self, alpha):
        self.dim_s, self.dim_x, self.dim_u = 3, 9, 2
        self._delta = alpha
        a = destroy(3)
        H0 = alpha * proj(3, 2)
        HX = 0.5 * (a.conj().T + a)
        HY = 0.5j * (a.conj().T - a)
        self.H_list = [H0, HX, HY]
        self.QE = self._QE(H0, [HX, HY])


class RWA_Transmon_Reduced(RWA_Transmon):
    """tests/util_qubits.py:119-138: same plant, observed only in the qubit block."""
    _QE = QExperiment32


class RWA_Crosstalk:
    """tests/util_qubits.py:39-57: H0 = xi/2 sz(x)sz; H1 = [sx(x)I / 2, I(x)sy / 2]."""

    def __init__(self, crosstalk):
        self.dim_u, self.dim_s, self.dim_x = 2, 4, 16
        self.crosstalk = crosstalk
        H0 = 0.5 * crosstalk * np.kron(SZ, SZ)
        H_x1 = 0.5 * np.kron(SX, I2)
        H_x2 = 0.5 * np.kron(I2, SY)
        self.H_list = [H0, H_x1, H_x2]
        self.H_list_1 = [0 * I2, SX]
        self.H_list_2 = [0 * I2, SY]
        self.QE = QCoupledExperiment(H0, [H_x1, H_x2])


class RWA_Coupled:
    """tests/util_qubits.py:19-36: H0 = sz(x)sz; controls sy(x)I, I(x)sy, sz(x)I."""

    def __init__(self):
        self.dim_u, self.dim_s, self.dim_x = 3, 4, 16
        self.H_list = [np.kron(SZ, SZ), np.kron(SY, I2), np.kron(I2, SY), np.kron(SZ, I2)]
        self.QE = QExperiment(self.H_list[0], self.H_list[1:])


def _pack(**kw):
    return kw


def config_qubit(order=1, discretize=None):
    """BASELINE config 1 (tests/test_mpc4quantum.py:607-670): ideal qubit |0> -> |1>, 1 % detuned plant."""
    clock = StepClock(dt=1, horizon=10, n_steps=20)
    sat = 2 * np.pi * 0.1
    du = 0.5 * sat
    wq = 2 * np.pi * 4
    nominal = RWA_Qubit(wq, wq, wq)
    A_init = (discretize or discretize_homogeneous)([liouvillian(h) for h in nominal.H_list], clock.dt, order)
    plant = RWA_Qubit(wq * 0.99, wq, wq)
    Q = np.diag([1.0, 0, 0, 1.0])
    R = (1e-2 / sat ** 2) * np.eye(1)
    Rx = rx(1e-4)
    rho0 = Rx @ proj(2, 0) @ Rx.conj().T
    target = proj(2, 1).reshape(-1)
    S, H = clock.n_steps, clock.horizon
    return _pack(name='qubit', x0=rho0.reshape(-1), dim_u=1, order=order,
                 X_targ=np.tile(target[:, None], (1, S + H + 1)), U_targ=np.zeros((1, S + H)),
                 clock=clock, experiment=plant.QE, model=_dmdc(A_init, 4), Q=Q, R=R, Qf=Q, sat=sat, du=du,
                 warm_start=True, target=target, wq=wq, nominal=nominal)


def config_transmon(order=1, horizon=16, n_steps=20, discretize=None):
    """BASELINE config 3 (tests/test_mpc4quantum.py:504-564): 3-level transmon, DRAG-like state transfer."""
    clock = StepClock(dt=0.25, horizon=horizon, n_steps=n_steps)
    sat = 2 * np.pi * 0.25
    du = 0.5 * sat
    anharm = -2 * np.pi * 0.1 * (1 / clock.dt)
    qubit = RWA_Transmon(alpha=anharm)
    A_init = (discretize or discretize_homogeneous)([liouvillian(h) for h in qubit.H_list], clock.dt, order)
    Q = np.zeros((9, 9))
    Q[0, 0] = 1
    Q[4, 4] = 1
    R = (1e-3 / sat ** 2) * np.eye(2)
    Rx = rx(1e-4)
    rho0 = proj(3, 0)
    rho0[:2, :2] = Rx.conj().T @ rho0[:2, :2] @ Rx
    target = proj(3, 1).reshape(-1)
    S, H = clock.n_steps, clock.horizon
    return _pack(name='transmon', x0=rho0.reshape(-1), dim_u=2, order=order,
                 X_targ=np.tile(target[:, None], (1, S + H + 1)), U_targ=np.zeros((2, S + H)),
                 clock=clock, experiment=qubit.QE, model=_dmdc(A_init, 9), Q=Q, R=R, Qf=Q, sat=sat, du=du,
                 warm_start=True, target=target, anharm=anharm, nominal=qubit)


def config_crosstalk(crosstalk=0.0, wiring='consistent', n_steps=50, discretize=None):
    """BASELINE config 4 (tests/test_mpc4quantum.py:281-368): two qubits, stacked 8-dim model, 16-dim plant.

    The reference test wires the model and the plant inconsistently (SURVEY.md section 4): the model's first
    control drives qubit 2 with sy and omits the 1/2.  ``wiring='consistent'`` (default) builds the model from
    the plant's own single-qubit generators (u0 -> sx/2 on qubit A, u1 -> sy/2 on qubit B);
    ``wiring='reference'`` reproduces the test literally.  ``discretize`` replaces the device discretisation
    (used by the CPU oracle, which has no GPU).
    """
    clock = StepClock(dt=0.5, horizon=20, n_steps=n_steps)
    clock.measure_freq = 2
    sat = 2 * np.pi * 0.1
    du = 0.25
    qubits = RWA_Crosstalk(crosstalk)
    Z4 = np.zeros((4, 4), dtype=complex)

    def blk(a, b):
        return np.block([[a, Z4], [Z4, b]])
    if wiring == 'reference':
        L1 = [liouvillian(h) for h in qubits.H_list_1]
        L2 = [liouvillian(h) for h in qubits.H_list_2]
        A_cts = [blk(L1[0], L2[0]), blk(Z4, L2[1]), blk(L1[1], Z4)]
    else:
        A_cts = [blk(Z4, Z4), blk(liouvillian(0.5 * SX), Z4), blk(Z4, liouvillian(0.5 * SY))]
    A_dst = (discretize or discretize_homogeneous)(A_cts, clock.dt, 1)
    r1, r2 = rx(-1e-3), rx(1e-3)
    rho1_init = r1 @ proj(2, 0) @ r1.conj().T
    rho2_init = r2 @ proj(2, 0) @ r2.conj().T
    x0 = np.kron(rho1_init, rho2_init).reshape(-1)
    target_model = np.concatenate([proj(2, 1).reshape(-1), proj(2, 0).reshape(-1)])
    target_plant = np.kron(proj(2, 1), proj(2, 0)).reshape(-1)
    q = np.diag([1.0, 0, 0, 1.0])
    Q = np.block([[q, np.zeros((4, 4))], [np.zeros((4, 4)), q]])
    R = 1e-3 * np.eye(2)
    S, H = clock.n_steps, clock.horizon
    return _pack(name='crosstalk', x0=x0, dim_u=2, order=1,
                 X_targ=np.tile(target_model[:, None], (1, S + H + 1)), U_targ=np.zeros((2, S + H)),
                 clock=clock, experiment=qubits.QE, model=_dmdc(A_dst, 8), Q=Q, R=R, Qf=Q, sat=sat, du=du,
                 warm_start=False, target=target_plant, nominal=qubits, kind='coupled')


def config_qubit_freq(order=1, n_steps=100, discretize=None):
    """tests/test_mpc4quantum.py:705-768 (test_NOT_state_freq): the qubit of config 1 with dt = 0.2, H = 50 and one
    plant measurement every 5 MPC steps (model steps in between, mpc.py:252-267)."""
    clock = StepClock(dt=0.2, horizon=50, n_steps=n_steps)
    clock.measure_freq = 5
    sat = 2 * np.pi * 0.1
    du = 0.1 * sat
    wq = 2 * np.pi * 4
    nominal = RWA_Qubit(wq, wq, wq)
    A_init = (discretize or discretize_homogeneous)([liouvillian(h) for h in nominal.H_list], clock.dt, order)
    plant = RWA_Qubit(wq * 0.99, wq, wq)
    Q = np.diag([1.0, 0, 0, 1.0])
    R = 1e-2 * np.eye(1)
    Rx = rx(1e-4)
    rho0 = Rx @ proj(2, 0) @ Rx.conj().T
    target = proj(2, 1).reshape(-1)
    S, H = clock.n_steps, clock.horizon
    return _pack(name='qubit_freq', x0=rho0.reshape(-1), dim_u=1, order=order,
                 X_targ=np.tile(target[:, None], (1, S + H + 1)), U_targ=np.zeros((1, S + H)),
                 clock=clock, experiment=plant.QE, model=_dmdc(A_init, 4), Q=Q, R=R, Qf=Q, sat=sat, du=du,
                 warm_start=True, target=target, wq=wq, nominal=nominal)


def config_cnot(n_steps=200, horizon=50, ramp_steps=None, discretize=None):
    """tests/test_mpc4quantum.py:399-466 (test_CNOT_state): two coupled qubits, fully vectorised 16-dim density
    matrix, three controls, ramped target (so the lagging target windows of mpc.py:276-277 matter)."""
    clock = StepClock(dt=0.25, horizon=horizon, n_steps=n_steps)
    sat = 2 * np.pi * 0.05
    du = 1 * sat
    qubits = RWA_Coupled()
    A_init = (discretize or discretize_homogeneous)([liouvillian(h) for h in qubits.H_list], clock.dt, 1)
    Rx1, Rx2 = rx(-1e-2), rx(1e-2)
    rho0 = np.kron(Rx1 @ proj(2, 0) @ Rx1.conj().T, Rx2 @ proj(2, 0) @ Rx2.conj().T)
    target = np.kron(proj(2, 0), proj(2, 1)).reshape(-1)
    S, H = clock.n_steps, clock.horizon
    ramp = ramp_steps or S
    incline = np.array([min(1.0, 2 * n / ramp) for n in range(S + H + 1)])
    Q = np.zeros((16, 16))
    for i in (0, 5, 10, 15):
        Q[i, i] = 1
    R = 1e-3 * np.eye(3)
    return _pack(name='cnot', x0=rho0.reshape(-1), dim_u=3, order=1,
                 X_targ=target[:, None] * incline[None, :], U_targ=np.zeros((3, S + H)),
                 clock=clock, experiment=qubits.QE, model=_dmdc(A_init, 16), Q=Q, R=R, Qf=Q, sat=sat, du=du,
                 warm_start=True, target=target, nominal=qubits)


def config_transmon_reduced(n_steps=20, horizon=10, discretize=None):
    """A two-level model (controls sx/2, sy/2) steering the three-level transmon of config 3 observed only in its
    qubit block (QExperiment32, experiment.py:215-235; util_qubits.py:119-138)."""
    clock = StepClock(dt=0.25, horizon=horizon, n_steps=n_steps)
    sat = 2 * np.pi * 0.25
    du = 0.5 * sat
    anharm = -2 * np.pi * 0.1 * (1 / clock.dt)
    plant = RWA_Transmon_Reduced(alpha=anharm)
    H_model = [0 * I2, 0.5 * SX, 0.5 * SY]
    A_init = (discretize or discretize_homogeneous)([liouvillian(h) for h in H_model], clock.dt, 1)
    Q = np.diag([1.0, 0, 0, 1.0])
    R = (1e-3 / sat ** 2) * np.eye(2)
    Rx = rx(1e-4)
    rho0 = proj(3, 0)
    rho0[:2, :2] = Rx.conj().T @ rho0[:2, :2] @ Rx
    target = proj(2, 1).reshape(-1)
    S, H = clock.n_steps, clock.horizon
    return _pack(name='transmon_reduced', x0=rho0.reshape(-1), dim_u=2, order=1,
                 X_targ=np.tile(target[:, None], (1, S + H + 1)), U_targ=np.zeros((2, S + H)),
                 clock=clock, experiment=plant.QE, model=_dmdc(A_init, 4), Q=Q, R=R, Qf=Q, sat=sat, du=du,
                 warm_start=True, target=target, nominal=plant, kind='trunc32')


def config_transmon_exact(horizon=16, n_steps=20):
    """Config 3 with the exact-discretisation model (``ExactModel``: x+ = expm(G(u) dt) x) in place of the Taylor
    blocks; everything else as ``config_transmon``."""
    from .model import ExactModel
    cfg = config_transmon(1, horizon=horizon, n_steps=n_steps, discretize=lambda L, dt, o: np.hstack([np.eye(9)] * 3))
    cfg['model'] = ExactModel([liouvillian(h) for h in cfg['nominal'].H_list], cfg['clock'].dt)
    cfg['name'] = 'transmon_exact'
    return cfg


def config_not_gate(order=1, n_steps=50, discretize=None):
    """tests/test_mpc4quantum.py:48-97 (test_NOT_gate): synthesis of the NOT gate on a resonant qubit, observed
    through the 16-dim process vector vec(U (x) U^*); dt = 0.05, H = 15, one control, identity costs, reference control
    0.5.  The reference test passes a target of only H + 1 columns (and keyword names RWA_Qubit does not have); here the
    target covers the whole run.  ``exit_condition`` is the test's callback, ``exit_infidelity`` the equivalent
    threshold on 1 - |tr(Uf^+ U)|^2 / 4:  ||p - pf||^2 = 8 (1 - F)."""
    from .experiment import QProcess
    clock = StepClock(dt=0.05, horizon=15, n_steps=n_steps)
    sat, du = 1.0, 0.25
    qubit = RWA_Qubit(np.pi, np.pi, np.pi)
    eye2, eye4 = np.eye(2), np.eye(4)
    As_cts = [-1j * np.kron(np.kron(h, eye2) - np.kron(eye2, h.conj()), eye4) for h in qubit.H_list]
    A_init = (discretize or discretize_homogeneous)(As_cts, clock.dt, order)
    U0 = rx(1e-3)
    p0 = np.kron(U0, U0.conj()).flatten()
    pf = np.kron(SX, SX.conj()).flatten()
    Q = np.eye(16)
    S, H = clock.n_steps, clock.horizon

    def exit_condition(p2, p1, u1):
        return ((p1 - pf).conj().T @ Q @ (p1 - pf)).real < 1e-2

    return _pack(name='not_gate', x0=p0, dim_u=1, order=order, X_targ=np.tile(pf[:, None], (1, S + H + 1)),
                 U_targ=0.5 * np.ones((1, S + H)), clock=clock, experiment=QProcess(qubit.H_list[0], [qubit.H_list[1]]),
                 model=_dmdc(A_init, 16), Q=Q, R=1e-2 * np.eye(1), Qf=10.0 * Q, sat=sat, du=du, warm_start=True,
                 target=pf / 4.0, kind='process', exit_condition=exit_condition, exit_infidelity=1e-2 / 8.0,
                 nominal=qubit, u0=U0.flatten())


def _ket_op(d, i, j):
    """|i><j| + |j><i| (symmetric part of one transition) on a d-level system."""
    out = np.zeros((d, d), dtype=complex)
    out[i, j] = out[j, i] = 1
    return out


def _y_op(d, i, j):
    """-i |i><j| + i |j><i| (the quadrature of _ket_op)."""
    out = np.zeros((d, d), dtype=complex)
    out[i, j], out[j, i] = -1j, 1j
    return out


# (dim_x, dim_u) pairs that have a configuration in config_shape (every compiled pair the BASELINE configs leave out)
NEW_SHAPES = ((4, 3), (4, 4), (8, 1), (8, 3), (8, 4), (9, 1), (9, 3), (9, 4), (16, 2), (16, 4))


def config_shape(c, m, order=1, n_steps=None, discretize=None):
    """A configuration for each pair of NEW_SHAPES, with the clock and cost conventions of the BASELINE config of the
    same state dimension.  ``cfg['detuning']`` is the plant operator ``ensemble_shape`` perturbs with.

      (4, 3)   qubit with sx/2, sy/2, sz/2 controls (config_qubit's clock, costs and 1 % detuned plant)
      (4, 4)   transmon with X01/2, Y01/2, a^+a and X12/2 drives, observed in its qubit block (QExperiment32); the model
               is the qubit block, where X12 does not act (config_transmon_reduced)
      (8, 1)   two qubits under ZZ crosstalk with one global X drive, both driven to |1> (config_crosstalk)
      (8, 3)   the same with X_A, Y_A, X_B;  (8, 4): X and Y on each qubit; qubit A to |1>, B stays in |0>
      (9, 1)   transmon driven on the X quadrature only (config_transmon)
      (9, 3)   transmon with X, Y and a detuning (a^+a) control;  (9, 4): qutrit with X01, Y01, X12, Y12 drives
      (16, 2)  NOT-gate synthesis with both quadratures (config_not_gate, run for n_steps without the exit test)
      (16, 4)  two-qubit density matrix with X and Y on each qubit under ZZ, ramped target (config_cnot)
    """
    if (c, m) not in NEW_SHAPES:
        raise ValueError('no configuration for (dim_x, dim_u) = (%d, %d)' % (c, m))
    disc = discretize or discretize_homogeneous
    name = 'shape_%d_%d' % (c, m)
    if c == 4 and m == 3:
        cfg = config_qubit(order, discretize=disc)
        wq = cfg['wq']
        H_model = [0 * SZ, 0.5 * SX, 0.5 * SY, 0.5 * SZ]
        cfg['model'] = _dmdc(disc([liouvillian(h) for h in H_model], cfg['clock'].dt, order), 4)
        cfg['experiment'] = QExperiment(-0.005 * wq * SZ, H_model[1:])
        cfg['R'] = cfg['R'][0, 0] * np.eye(3)
        det = 0.5 * SZ
    elif c == 4:
        cfg = config_transmon_reduced(discretize=disc)
        alpha = cfg['nominal']._delta
        num = destroy(3).conj().T @ destroy(3)
        cfg['experiment'] = QExperiment32(alpha * proj(3, 2), [0.5 * _ket_op(3, 0, 1), 0.5 * _y_op(3, 0, 1), num,
                                                                0.5 * _ket_op(3, 1, 2)])
        H_model = [0 * I2, 0.5 * SX, 0.5 * SY, proj(2, 1), 0 * I2]
        cfg['model'] = _dmdc(disc([liouvillian(h) for h in H_model], cfg['clock'].dt, order), 4)
        cfg['R'] = cfg['R'][0, 0] * np.eye(4)
        cfg['target'] = proj(3, 1).reshape(-1)      # fidelity of the plant state, which is a qutrit
        det = num
    elif c == 8:
        cfg = config_crosstalk(0.05, discretize=disc)
        Z4 = np.zeros((4, 4), dtype=complex)

        def blk(a, b):
            return np.block([[a, Z4], [Z4, b]])
        LX, LY = liouvillian(0.5 * SX), liouvillian(0.5 * SY)
        XA, YA, XB, YB = (0.5 * np.kron(SX, I2), 0.5 * np.kron(SY, I2), 0.5 * np.kron(I2, SX), 0.5 * np.kron(I2, SY))
        drives = {1: ([blk(LX, LX)], [XA + XB]), 3: ([blk(LX, Z4), blk(LY, Z4), blk(Z4, LX)], [XA, YA, XB]),
                  4: ([blk(LX, Z4), blk(LY, Z4), blk(Z4, LX), blk(Z4, LY)], [XA, YA, XB, YB])}[m]
        cfg['model'] = _dmdc(disc([blk(Z4, Z4)] + drives[0], cfg['clock'].dt, order), 8)
        cfg['experiment'] = QCoupledExperiment(cfg['experiment'].H0, drives[1])
        cfg['R'] = 1e-3 * np.eye(m)
        if m == 1:      # one global drive flips both qubits
            S, H = cfg['clock'].n_steps, cfg['clock'].horizon
            target_model = np.concatenate([proj(2, 1).reshape(-1)] * 2)
            cfg['X_targ'] = np.tile(target_model[:, None], (1, S + H + 1))
            cfg['target'] = np.kron(proj(2, 1), proj(2, 1)).reshape(-1)
            # both qubits start tilted the same way: with config_crosstalk's opposite tilts the first-order effects of
            # the one drive on the two populations cancel, the first QP sits on a saddle at u = 0 and a relative
            # perturbation of 1e-15 in the model moves the closed loop's controls by 0.25
            r = rx(-1e-3)
            rho = r @ proj(2, 0) @ r.conj().T
            cfg['x0'] = np.kron(rho, rho).reshape(-1)
        det = 0.5 * (np.kron(SZ, I2) + np.kron(I2, SZ))
    elif c == 9:
        cfg = config_transmon(order, discretize=disc)
        H0 = cfg['nominal'].H_list[0]
        HX, HY = cfg['nominal'].H_list[1:]
        num = destroy(3).conj().T @ destroy(3)
        H1 = {1: [HX], 3: [HX, HY, num],
              4: [0.5 * _ket_op(3, 0, 1), 0.5 * _y_op(3, 0, 1), 0.5 * _ket_op(3, 1, 2), 0.5 * _y_op(3, 1, 2)]}[m]
        cfg['model'] = _dmdc(disc([liouvillian(h) for h in [H0] + H1], cfg['clock'].dt, order), 9)
        cfg['experiment'] = QExperiment(H0, H1)
        cfg['R'] = cfg['R'][0, 0] * np.eye(m)
        det = num
    elif m == 2:
        from .experiment import QProcess
        cfg = config_not_gate(order, discretize=disc)
        H_list = [0 * SZ, 0.5 * SX, 0.5 * SY]
        eye2, eye4 = np.eye(2), np.eye(4)
        As_cts = [-1j * np.kron(np.kron(h, eye2) - np.kron(eye2, h.conj()), eye4) for h in H_list]
        cfg['model'] = _dmdc(disc(As_cts, cfg['clock'].dt, order), 16)
        cfg['experiment'] = QProcess(H_list[0], H_list[1:])
        cfg['U_targ'] = np.vstack([cfg['U_targ'], np.zeros_like(cfg['U_targ'])])
        cfg['R'] = 1e-2 * np.eye(2)
        for key in ('exit_condition', 'exit_infidelity'):
            cfg.pop(key)
        det = 0.5 * SZ
    else:
        cfg = config_cnot(n_steps=n_steps or 200, discretize=disc)
        H0 = np.kron(SZ, SZ)
        H1 = [np.kron(SX, I2), np.kron(SY, I2), np.kron(I2, SX), np.kron(I2, SY)]
        cfg['model'] = _dmdc(disc([liouvillian(h) for h in [H0] + H1], cfg['clock'].dt, order), 16)
        cfg['experiment'] = QExperiment(H0, H1)
        cfg['R'] = 1e-3 * np.eye(4)
        det = 0.5 * (np.kron(SZ, I2) + np.kron(I2, SZ))
    if cfg['U_targ'].shape[0] != m:     # every control but the NOT gate's tracks zero
        cfg['U_targ'] = np.zeros((m, cfg['U_targ'].shape[1]))
    cfg.update(name=name, dim_u=m, order=order, detuning=det)
    if n_steps is not None and n_steps != cfg['clock'].n_steps:
        clock = cfg['clock']
        new = StepClock(dt=clock.dt, horizon=clock.horizon, n_steps=n_steps)
        new.measure_freq = clock.measure_freq
        cfg['clock'] = new
        cols = n_steps + clock.horizon + 1
        cfg['X_targ'] = _fit_columns(cfg['X_targ'], cols)
        cfg['U_targ'] = _fit_columns(cfg['U_targ'], cols - 1)
    return cfg


def _fit_columns(a, n):
    """The first n columns of a, the last one repeated when a has fewer."""
    if a.shape[1] >= n:
        return a[:, :n]
    return np.hstack([a, np.repeat(a[:, -1:], n - a.shape[1], axis=1)])


def _dmdc(A_full, c):
    p = A_full.shape[1] // c - 1
    return DMDc(c, c, c * p, A_full)


def mpc_args(cfg):
    """Positional/keyword arguments for mpc()/mpc_ensemble() from a config dict."""
    args = (cfg['x0'], cfg['dim_u'], cfg['order'], cfg['X_targ'], cfg['U_targ'], cfg['clock'],
            cfg['experiment'], cfg['model'], cfg['Q'], cfg['R'], cfg['Qf'])
    kw = dict(sat=cfg['sat'], du=cfg['du'], warm_start=cfg['warm_start'], progress_bar=False)
    return args, kw


# ----------------------------------------------------------------------------
# Ensembles of perturbed plants (SURVEY.md section 8(d)); drawn on the host from a fixed seed so that the
# members are independent of the GPU count.  Returned arrays: H0 [N, d, d], H1 [N, m, d, d] complex128.
# ----------------------------------------------------------------------------
ENSEMBLE_SEED = 20220113


class _Draws:
    """The ensemble's uniform draws, or only members [lo, hi) of them, bit for bit the same either way.

    The full ensemble is a sequence of length-N ``rng.uniform`` arrays from ``np.random.default_rng(seed)``.  Each
    double consumes one 64-bit output of PCG64, so member k of the j-th array is output j N + k of the stream:
    ``bit_generator.advance`` jumps there, and a rank draws its own shard without materialising the other members
    (1 M members x 8 ranks would otherwise hold 432 MB each)."""

    def __init__(self, seed, N, lo=None, hi=None):
        self.seed, self.N = seed, int(N)
        self.lo, self.hi = (0, self.N) if lo is None else (int(lo), int(hi))
        self.count = 0

    def uniform(self, a, b):
        rng = np.random.default_rng(self.seed)
        rng.bit_generator.advance(self.count * self.N + self.lo)
        self.count += 1
        return rng.uniform(a, b, self.hi - self.lo)


def ensemble_qubit(N, seed=ENSEMBLE_SEED, wq=2 * np.pi * 4, lo=None, hi=None):
    """C2: detuning scale s ~ U[0.98, 1.02] (plant H0 = (s-1) wq sz / 2), amplitude scale a ~ U[0.9, 1.1].
    lo, hi: only members [lo, hi) of the N-member ensemble (same values as slicing the full draw)."""
    rng = _Draws(seed, N, lo, hi)
    s = rng.uniform(0.98, 1.02)
    a = rng.uniform(0.9, 1.1)
    H0 = 0.5 * ((s - 1) * wq)[:, None, None] * SZ
    H1 = (a[:, None, None] * (0.5 * SX))[:, None]
    return EnsembleQExperiment(H0, H1), dict(detuning_scale=s, amplitude_scale=a)


def ensemble_transmon(N, seed=ENSEMBLE_SEED, dt=0.25, lo=None, hi=None):
    """C3/C5: anharmonicity scale ~U[0.9,1.1], amplitude scale ~U[0.9,1.1], detuning ~U[-0.02,0.02] 2pi/dt on a^+a.
    lo, hi: only members [lo, hi) of the N-member ensemble (same values as slicing the full draw)."""
    rng = _Draws(seed, N, lo, hi)
    k = rng.uniform(0.9, 1.1)
    a_s = rng.uniform(0.9, 1.1)
    det = rng.uniform(-0.02, 0.02) * 2 * np.pi / dt
    alpha = -2 * np.pi * 0.1 / dt
    a = destroy(3)
    num = a.conj().T @ a
    HX = 0.5 * (a.conj().T + a)
    HY = 0.5j * (a.conj().T - a)
    H0 = (k * alpha)[:, None, None] * proj(3, 2) + det[:, None, None] * num
    H1 = np.stack([a_s[:, None, None] * HX, a_s[:, None, None] * HY], axis=1)
    return EnsembleQExperiment(H0, H1), dict(anharm_scale=k, amplitude_scale=a_s, detuning=det)


def ensemble_crosstalk(N, seed=ENSEMBLE_SEED, lo=None, hi=None):
    """C4: ZZ strength xi ~ U[0, 2pi 0.02], amplitude scale ~U[0.9,1.1]; plant observed through partial traces.
    lo, hi: only members [lo, hi) of the N-member ensemble (same values as slicing the full draw)."""
    rng = _Draws(seed, N, lo, hi)
    xi = rng.uniform(0, 2 * np.pi * 0.02)
    a_s = rng.uniform(0.9, 1.1)
    H0 = 0.5 * xi[:, None, None] * np.kron(SZ, SZ)
    H1 = np.stack([a_s[:, None, None] * (0.5 * np.kron(SX, I2)), a_s[:, None, None] * (0.5 * np.kron(I2, SY))],
                  axis=1)
    return EnsembleQExperiment(H0, H1, kind='coupled'), dict(xi=xi, amplitude_scale=a_s)


def ensemble_not_gate(N, seed=ENSEMBLE_SEED, lo=None, hi=None):
    """Gate-synthesis ensemble: residual detuning delta_k ~ U[-0.05, 0.05] * 2 pi (H0 = delta_k sigma_z / 2) and drive
    amplitude scale a_k ~ U[0.9, 1.1] (H1 = a_k sigma_x / 2)."""
    from .experiment import EnsembleQExperiment
    rng = _Draws(seed, N, lo, hi)
    delta = rng.uniform(-0.05, 0.05) * 2 * np.pi
    amp = rng.uniform(0.9, 1.1)
    H0 = 0.5 * delta[:, None, None] * SZ[None]
    H1 = (0.5 * amp[:, None, None] * SX[None])[:, None]
    return EnsembleQExperiment(H0, H1, kind='process'), dict(delta=delta, amp=amp)


def ensemble_shape(cfg, N, seed=ENSEMBLE_SEED, lo=None, hi=None):
    """Ensemble of a ``config_shape`` plant: every drive amplitude scaled by a ~ U[0.9, 1.1] and a detuning
    delta ~ U[-0.1, 0.1] sat added to H0 along ``cfg['detuning']``.
    lo, hi: only members [lo, hi) of the N-member ensemble (same values as slicing the full draw)."""
    rng = _Draws(seed, N, lo, hi)
    a = rng.uniform(0.9, 1.1)
    det = rng.uniform(-0.1, 0.1) * cfg['sat']
    ex = cfg['experiment']
    H0 = ex.H0[None] + det[:, None, None] * cfg['detuning'][None]
    H1 = a[:, None, None, None] * np.stack(ex.H1_list)[None]
    return EnsembleQExperiment(H0, H1, kind=cfg.get('kind', 'identity')), dict(amplitude_scale=a, detuning=det)


def transmon_model_liouvillians(N, seed=ENSEMBLE_SEED + 1, dt=0.25, lo=None, hi=None):
    """Perturbed controller MODELS for the transmon (pure numpy): member k believes in the anharmonicity
    k_k alpha, k_k ~ U[0.95, 1.05], and in drive amplitudes scaled by g_k ~ U[0.97, 1.03].
    Returns the Liouvillians L [N, 3, 9, 9] of [H0, HX, HY] per member (row-major vec(rho)) and the draws."""
    rng = _Draws(seed, N, lo, hi)
    k = rng.uniform(0.95, 1.05)
    g = rng.uniform(0.97, 1.03)
    N = len(k)
    alpha = -2 * np.pi * 0.1 / dt
    a = destroy(3)
    H = np.stack([(k * alpha)[:, None, None] * proj(3, 2)[None],
                  g[:, None, None] * (0.5 * (a.conj().T + a))[None],
                  g[:, None, None] * (0.5j * (a.conj().T - a))[None]], axis=1)          # [N, 3, 3, 3]
    eye = np.eye(3)
    L = -1j * (np.einsum('nkab,cd->nkacbd', H, eye) - np.einsum('ab,nkdc->nkacbd', eye, H)).reshape(N, 3, 9, 9)
    return L, dict(model_anharm_scale=k, model_amplitude_scale=g)


def ensemble_transmon_models(N, order=1, dt=0.25, seed=ENSEMBLE_SEED + 1, lo=None, hi=None):
    """The N perturbed models discretised on the device (m4q_taylor_discretize_batched, vectorize.py:8-49 per member)
    as a ``DMDcEnsemble`` for ``mpc_ensemble``."""
    from .model import DMDcEnsemble
    from .vectorize import discretize_homogeneous_batched
    L, params = transmon_model_liouvillians(N, seed, dt, lo, hi)
    A = discretize_homogeneous_batched(L, dt, order)
    return DMDcEnsemble(9, 9, A.shape[2] - 9, A), params
