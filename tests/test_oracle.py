"""CPU tests of the oracle (oracle/restate.py, oracle/admm_model.py) against the fixtures generated from the
reference's own code (oracle/make_golden.py).  No GPU, no /root/reference needed."""
import itertools
import math
import os

import numpy as np
import pytest

from oracle import restate as rs, admm_model as am, refshim
from mpc4quantum_b200 import linearize, systems
from conftest import load_golden


def test_power_table_matches_reference_order():
    # SURVEY 3.2: for dim_u = 2, order = 2 the reference orders u1, u1^2, u2, u1 u2, u2^2
    assert rs.power_table(2, 2).tolist() == [[0, 0], [1, 0], [2, 0], [0, 1], [1, 1], [0, 2]]
    assert rs.power_table(1, 3).tolist() == [[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]]


@pytest.mark.parametrize('tag,orders', [('qubit', (1, 2, 3)), ('transmon', (1, 2, 3)), ('coupled', (1, 2))])
def test_taylor_discretize_vs_reference(unit_golden, tag, orders):
    L = list(unit_golden['disc_%s_L' % tag])
    dt = float(unit_golden['disc_%s_dt' % tag])
    for o in orders:
        assert np.abs(rs.taylor_discretize(L, dt, o) - unit_golden['disc_%s_o%d' % (tag, o)]).max() < 1e-13


def test_reference_test_discretization_case():
    """The reference's only live hot-path assertion (tests/test_mpc4quantum.py:182-188): order 1, dt = 1."""
    rng = np.random.default_rng(0)
    A, N1, N2 = (rng.normal(size=(8, 8)) + 1j * rng.normal(size=(8, 8)) for _ in range(3))
    out = rs.taylor_discretize([A, N1, N2], 1.0, 1)
    assert np.allclose(out, np.hstack([np.eye(8) + A, N1, N2]))


def test_vectorize_me_restatement(unit_golden):
    out = rs.liouvillian_in_basis(unit_golden['vecme_H'], list(unit_golden['vecme_basis']))
    assert np.abs(out - unit_golden['vecme_out']).max() < 1e-13


@pytest.mark.parametrize('tag,m', [('qubit', 1), ('transmon', 2), ('transmon1', 2), ('coupled', 3)])
def test_linearisation_vs_reference(unit_golden, tag, m):
    bm = rs.BilinearModel(unit_golden['lin_%s_A_full' % tag], m, int(unit_golden['lin_%s_order' % tag]))
    X, U = unit_golden['lin_%s_X' % tag], unit_golden['lin_%s_U' % tag]
    A, B, D = bm.along(X, U, U.shape[1])
    assert np.abs(np.array(A) - unit_golden['lin_%s_A' % tag]).max() < 1e-12
    assert np.abs(np.array(B) - unit_golden['lin_%s_B' % tag]).max() < 1e-12
    assert np.abs(np.array(D) - unit_golden['lin_%s_D' % tag]).max() < 1e-11
    # Delta_t == -B_t u_t identically (SURVEY 3.2) and the Jacobian agrees with central differences
    assert np.abs(np.array(D) + np.einsum('tij,jt->ti', np.array(B), U)).max() < 1e-11
    eps = 1e-6
    e0 = np.zeros(m)
    e0[0] = eps
    fd = (bm.step(X[:, 2], U[:, 2] + e0) - bm.step(X[:, 2], U[:, 2] - e0)) / (2 * eps)
    assert np.abs(fd - B[2][:, 0]).max() < 1e-7


@pytest.mark.parametrize('tag', ['qubit', 'transmon', 'transmon_full', 'cross'])
def test_line_search_quirk_vs_reference(unit_golden, tag):
    X, U = unit_golden['ls_%s_X' % tag], unit_golden['ls_%s_U' % tag]
    a, s = rs.line_search(list(unit_golden['ls_%s_Q' % tag]), list(unit_golden['ls_%s_R' % tag]), X[0], U[0], X[1], U[1],
                          X[2], U[2])
    assert abs(a - float(unit_golden['ls_%s_alpha' % tag])) < 1e-12
    assert abs(s - float(unit_golden['ls_%s_step' % tag])) < 1e-10


def test_partial_trace_and_kron(unit_golden):
    """The reference's test_partialTrace (tests/test_mpc4quantum.py:190-213) restated: product states round-trip."""
    assert np.abs(rs.lift_coupled(unit_golden['lift_rho']) - unit_golden['lift_out']).max() < 1e-14
    assert np.abs(rs.proj_coupled(unit_golden['lift_out']) - unit_golden['proj_out']).max() < 1e-14
    rng = np.random.default_rng(1)
    a = rng.normal(size=(2, 2)) + 1j * rng.normal(size=(2, 2))
    b = rng.normal(size=(2, 2)) + 1j * rng.normal(size=(2, 2))
    a, b = a @ a.conj().T, b @ b.conj().T
    a, b = a / np.trace(a), b / np.trace(b)
    stacked = rs.lift_coupled(np.kron(a, b).reshape(-1))
    assert np.allclose(stacked, np.concatenate([a.reshape(-1), b.reshape(-1)]))
    assert np.allclose(rs.proj_coupled(stacked), np.kron(a, b).reshape(-1))


@pytest.mark.parametrize('tag', ['qubit', 'transmon', 'cross'])
def test_qp_oracles_agree_and_are_kkt_certified(qp_golden, tag):
    """Exact active-set oracle == stored solutions; the numpy model of the device ADMM+polish lands on the same
    optimum; both carry a KKT certificate that does not depend on how the solution was found."""
    g = qp_golden
    H = g['%s_U' % tag].shape[2]
    for i in (0, 2, 5):
        args = (g['%s_x_init' % tag][i], g['%s_X_bm' % tag][i], g['%s_U_bm' % tag][i], [g['%s_Q' % tag]] * H + [g['%s_Qf' % tag]],
                [g['%s_R' % tag]] * H, list(g['%s_A' % tag][i]), list(g['%s_B' % tag][i]), list(g['%s_D' % tag][i]),
                g['%s_u_prev' % tag][i], float(g['%s_sat' % tag]), float(g['%s_du' % tag]))
        X, U, obj, info = rs.qp_exact(*args)
        assert np.abs(U - g['%s_U' % tag][i]).max() < 1e-10
        assert info['kkt'][0] < 1e-8 and info['kkt'][1] < 1e-12
        X2, U2, obj2, _ = am.qp_admm(*args, rho=0.1, eps=1e-2)
        assert np.abs(U2 - U).max() < 1e-9 and abs(obj2 - obj) < 1e-9 * max(1, abs(obj))
        kkt = rs.qp_kkt(info, U2)
        assert kkt[0] < 1e-8 and kkt[1] < 1e-12
        # a perturbed point is NOT certified: the certificate has teeth
        assert rs.qp_kkt(info, np.clip(U + 1e-3, -args[9], args[9]))[0] > 1e-6


def test_restated_loop_reproduces_reference_run():
    """oracle/restate.mpc_loop == the reference's mpc() (run through the shim when the fixture was made)."""
    g = load_golden('loop_qubit_o1')
    cfg = systems.config_qubit(1, discretize=rs.taylor_discretize)
    assert np.abs(cfg['model'].A - g['A_full']).max() < 1e-14
    plant = rs.ExpmPlant(cfg['experiment'].H0, cfg['experiment'].H1_list)
    stats = {}
    xs, us, ec = rs.mpc_loop(cfg['x0'], 1, 1, cfg['X_targ'], cfg['U_targ'], 1.0, 10, 20, plant, cfg['model'].A, cfg['Q'],
                             cfg['R'], cfg['Qf'], cfg['sat'], cfg['du'], stats=stats)
    assert ec == 0 and stats['qp_per_step'] == list(g['qp_per_step'])
    assert np.abs(us - g['us']).max() < 1e-6 and np.abs(xs - g['xs']).max() < 1e-6
    assert abs(float(np.real(xs[3, -1])) - 0.999479038) < 1e-8          # SURVEY 8c smoke value
    assert np.allclose(us[0, :3], [0.31416, 0.31416, 0.62832], atol=1e-5)


def test_loop_quirks_are_exercised_by_fixture():
    """measure_freq = 2, warm_start = False, lift/proj (crosstalk config): newest-first control window (mpc.py:257),
    lagging targets, model steps between measurements -- all of it inside the stored reference run."""
    g = load_golden('loop_crosstalk')
    cfg = systems.config_crosstalk(0.05, n_steps=4, discretize=rs.taylor_discretize)
    plant = rs.ExpmPlant(cfg['experiment'].H0, cfg['experiment'].H1_list, rs.lift_coupled, rs.proj_coupled)
    xs, us, ec = rs.mpc_loop(cfg['x0'], 2, 1, cfg['X_targ'], cfg['U_targ'], 0.5, 20, 4, plant, cfg['model'].A, cfg['Q'],
                             cfg['R'], cfg['Qf'], cfg['sat'], cfg['du'], warm_start=False, measure_freq=2)
    assert ec == 0
    assert np.abs(us - g['us'][:, :4]).max() < 1e-7 and np.abs(xs - g['xs'][:, :5]).max() < 1e-7
    # odd steps are model predictions pushed through proj: product states
    x1 = xs[:, 1]
    assert np.abs(rs.proj_coupled(rs.lift_coupled(x1)) - x1).max() < 1e-12


def _reference_monomial_order(L, dt, order, blocks, rng):
    """The monomial of each block of the reference's discretize_homogeneous output, read off the blocks themselves: the
    order-k Taylor polynomial of exp((L0 + sum u_i L_i) dt), formed by matrix powers, is sum_b phi_b(u) blocks[b], so a
    least-squares fit at random u gives phi_b(u) for every block, and each phi_b is matched to one exponent tuple."""
    m = len(L) - 1
    basis = blocks.reshape(len(blocks), -1).T
    us = rng.uniform(-1, 1, size=(3 * len(blocks), m))
    phi = []
    for u in us:
        G = (L[0] + sum(ui * Li for ui, Li in zip(u, L[1:]))) * dt
        T = sum(np.linalg.matrix_power(G, j) / math.factorial(j) for j in range(order + 1)).reshape(-1)
        x, _, rank, _ = np.linalg.lstsq(basis, T, rcond=None)
        assert rank == len(blocks) and np.abs(basis @ x - T).max() < 1e-12
        phi.append(x)
    phi = np.array(phi)
    candidates = [e for e in itertools.product(range(order + 1), repeat=m) if sum(e) <= order]
    found = []
    for b in range(len(blocks)):
        err = [np.abs(phi[:, b] - np.prod(us ** np.array(e), axis=1)).max() for e in candidates]
        assert min(err) < 1e-10, (b, min(err))
        found.append(list(candidates[int(np.argmin(err))]))
    return found


def test_shim_runs_reference_functions(unit_golden):
    """The control-monomial order of the reference (linearize.py:92-116) against power_table and the package's
    create_power_list, for dim_u = 1, 2, 3 and orders up to 3.  The order is recovered from the reference's own
    discretisation blocks (tests/golden/unit.npz); where the reference tree is present, also through the shim."""
    rng = np.random.default_rng(3)
    cases = 0
    for tag in ('qubit', 'transmon', 'coupled'):
        L, dt = list(unit_golden['disc_%s_L' % tag]), float(unit_golden['disc_%s_dt' % tag])
        c, m = L[0].shape[0], len(L) - 1
        for order in (1, 2, 3):
            key = 'disc_%s_o%d' % (tag, order)
            if key not in unit_golden:
                continue
            blocks = unit_golden[key].reshape(c, -1, c).transpose(1, 0, 2)
            found = _reference_monomial_order(L, dt, order, blocks, rng)
            assert found == rs.power_table(order, m).tolist(), (tag, order)
            assert found == [list(p) for p in linearize.create_power_list(order, m)], (tag, order)
            cases += 1
    assert cases == 8
    if refshim.available():
        lin = refshim.module('linearize')
        for order, m in ((2, 2), (3, 1), (3, 3)):
            assert [list(p) for p in lin.create_power_list(order, m)] == rs.power_table(order, m).tolist()


def test_process_maps_and_gate_loop_vs_reference():
    """Gate synthesis (experiment.py:336-417): the restated lift / proj / process propagation against the vectors of
    the reference's own QSynthesis statics, and the restated closed loop against the reference loop fixture."""
    g = load_golden('gate')
    for n in (2, 3):
        for U, p, b in zip(g['U%d' % n], g['lift%d' % n], g['proj%d' % n]):
            assert np.abs(rs.lift_process(U.reshape(-1)) - p).max() < 1e-15
            assert np.abs(rs.proj_process(p) - b).max() < 1e-14
    pl = rs.ProcessPlant(g['sim_H0'], list(g['sim_H1']))
    assert np.abs(pl.simulate(g['sim_P'][:, 0], g['sim_ts'], g['sim_u']) - g['sim_P']).max() < 1e-13
    gl = load_golden('loop_not_gate_o1_exit')
    cfg = systems.config_not_gate(1, n_steps=90, discretize=rs.taylor_discretize)
    assert np.abs(cfg['model'].A - gl['A_full']).max() < 1e-14
    stats = {}
    xs, us, ec = rs.mpc_loop(cfg['x0'], 1, 1, cfg['X_targ'], cfg['U_targ'], cfg['clock'].dt, cfg['clock'].horizon,
                             cfg['clock'].n_steps, rs.ProcessPlant(cfg['experiment'].H0, cfg['experiment'].H1_list),
                             cfg['model'].A, cfg['Q'], cfg['R'], cfg['Qf'], cfg['sat'], cfg['du'], stats=stats,
                             exit_condition=cfg['exit_condition'])
    assert ec == 1 == int(gl['exit_code'])
    assert xs.shape == gl['xs'].shape and us.shape == gl['us'].shape
    assert np.abs(us - gl['us']).max() < 1e-9 and np.abs(xs - gl['xs']).max() < 1e-9
    assert np.array_equal(stats['qp_per_step'], gl['qp_per_step'])
    # ||p - pf||^2 = 8 (1 - F): the callback of the reference test is a threshold on the gate infidelity
    p = gl['xs'][:, -1]
    pf = cfg['X_targ'][:, 0]
    assert abs(np.vdot(p - pf, p - pf).real - 8 * (1 - np.real(np.vdot(cfg['target'], p)))) < 1e-12


def test_exact_model_oracle_against_finite_differences(unit_golden):
    """The oracle of the exact-discretisation mode (an extension: no reference vectors exist) is pinned to first
    principles: A_t is the propagator of the step map, B_t its derivative w.r.t. the control (central difference),
    Delta_t closes the affine expansion, and for small dt the map tends to the reference's Taylor model."""
    from scipy.linalg import expm
    L = list(unit_golden['disc_transmon_L'])
    dt = float(unit_golden['disc_transmon_dt'])
    model = rs.ExactModel(L, dt)
    rng = np.random.default_rng(4)
    c, m, H = 9, 2, 5
    X = rng.normal(size=(c, H + 1)) + 1j * rng.normal(size=(c, H + 1))
    U = rng.uniform(-1.5, 1.5, size=(m, H))
    A_ls, B_ls, D_ls = model.along(X, U, H)
    for t in range(H):
        G = (L[0] + U[0, t] * L[1] + U[1, t] * L[2]) * dt
        assert np.abs(A_ls[t] - expm(G)).max() < 1e-14
        assert np.abs(model.step(X[:, t], U[:, t]) - A_ls[t] @ X[:, t]).max() < 1e-13
        for i in range(m):
            e = np.zeros(m)
            e[i] = 1e-6
            fd = (model.step(X[:, t], U[:, t] + e) - model.step(X[:, t], U[:, t] - e)) / 2e-6
            assert np.abs(B_ls[t][:, i] - fd).max() < 1e-8
        # affine expansion around (x_t, u_t): f(x_t, u_t) = A_t x_t + B_t u_t + Delta_t
        assert np.abs(A_ls[t] @ X[:, t] + B_ls[t] @ U[:, t] + D_ls[t] - model.step(X[:, t], U[:, t])).max() < 1e-13
    # consistency with the reference's discretisation: the order-k Taylor blocks are the expansion of the same map
    for order, tol in ((1, 0.3), (2, 0.05), (3, 0.01)):
        bm = rs.BilinearModel(unit_golden['disc_transmon_o%d' % order], m, order)
        u = 0.3 * U[:, 0]
        err = np.abs(bm.step(X[:, 0], u) - model.step(X[:, 0], u)).max() / np.abs(X[:, 0]).max()
        assert err < tol, (order, err)


def test_h100_order1_oracle_and_its_costate_multipliers():
    """BASELINE config 3 at H = 100, order 1 (tests/golden/qp_h100.npz, from the reference loop): the oracle re-solves
    the captured QPs to the recorded answer, and the last-resort active set -- multipliers taken from the costates of
    the sparse KKT solve instead of an adjoint sweep through prod A_t (noise floor eps ||prod A_t||^2) -- lands on the
    same optimum.  The costate gradient agrees with the adjoint gradient where the latter still has digits."""
    g = load_golden('qp_h100')
    H = g['h100_U'].shape[2]
    Q_ls, R_ls = [g['h100_Q']] * H + [g['h100_Qf']], [g['h100_R']] * H
    sat, du = float(g['h100_sat']), float(g['h100_du'])
    i = int(np.argmax(g['h100_step']))          # the mildest of them (step 9): seconds on one core
    args = (g['h100_x_init'][i], g['h100_X_bm'][i], g['h100_U_bm'][i], Q_ls, R_ls, list(g['h100_A'][i]),
            list(g['h100_B'][i]), list(g['h100_D'][i]), g['h100_u_prev'][i], sat, du)
    X, U, obj, info = rs.qp_exact(*args)
    assert np.abs(U - g['h100_U'][i]).max() < 1e-9
    prob, lo, hi = info['prob'], info['lo'], info['hi']
    X2, U2, g2 = rs._active_set_kkt_multipliers(prob, lo, hi)
    assert np.abs(U2.T - U).max() < 1e-7
    fixed = (U.T <= lo + 1e-13) | (U.T >= hi - 1e-13)
    vals = np.where(U.T <= lo + 1e-13, lo, hi)
    Xs, Us, gk = prob.solve_fixed(fixed, vals, want_grad=True)
    ga = prob.gradient(Xs, Us)
    assert np.abs(gk[~fixed]).max() < 1e-9                     # stationary on the free controls
    assert np.abs(gk - ga).max() < 1e-4 * max(1.0, np.abs(ga).max())
    # the loop fixture records how far two CPU evaluations of the same algorithm part, and the measured amplification
    loop = load_golden('loop_transmon_o1_h100')
    assert int(loop['exit_code']) == 0 and loop['us'].shape == (2, 20)
    assert loop['restatement_gap_us'][:12].max() < 1e-8 < loop['restatement_gap_us'][-1]
    assert loop['perturbation_gap_us'].shape == (3, 20)


def test_kkt_interior_point_model_of_the_device_solver():
    """oracle/kkt_model.py (the numpy statement of csrc/m4q_kkt.cuh: stage-ordered KKT system, pivoted LU, interior-point
    working set, refined polish) against the exact oracle: a random short QP with a full Hermitian cost, and the QP of
    step 9 of the reference loop at H = 100 with the order-1 model (||prod A_t|| = 5e7, 23 controls on a bound)."""
    from oracle import kkt_model as km
    rng = np.random.default_rng(5)
    c, m, H = 4, 2, 12

    def crandn(*shape):
        return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
    A_ls = [np.eye(c) + 0.2 * crandn(c, c) / np.sqrt(c) for _ in range(H)]
    B_ls = [0.4 * crandn(c, m) for _ in range(H)]
    D_ls = [0.05 * crandn(c, 1) for _ in range(H)]
    L = crandn(c, c) / np.sqrt(c)
    Q = L @ L.conj().T
    R = 0.05 * np.eye(m)
    args = (crandn(c), crandn(c, H + 1), 0.3 * rng.standard_normal((m, H)), [Q] * (H + 1), [R] * H, A_ls, B_ls, D_ls,
            0.3 * rng.standard_normal(m), 0.6, 0.25)
    X, U, obj, info = rs.qp_exact(*args)
    Uk, stats = km.qp_kkt_ipm(info['prob'], info['lo'], info['hi'])
    assert Uk is not None and stats['polish_rounds'] <= 3 and stats['ipm_solves'] <= 25
    assert np.abs(Uk.T - U).max() < 1e-9
    assert (np.abs(np.abs(U) - 0.6) < 1e-12).sum() >= 3          # the box is active in this instance
    g = load_golden('qp_h100')
    Hh = g['h100_U'].shape[2]
    i = int(np.argmax(g['h100_step']))
    args = (g['h100_x_init'][i], g['h100_X_bm'][i], g['h100_U_bm'][i], [g['h100_Q']] * Hh + [g['h100_Qf']],
            [g['h100_R']] * Hh, list(g['h100_A'][i]), list(g['h100_B'][i]), list(g['h100_D'][i]), g['h100_u_prev'][i],
            float(g['h100_sat']), float(g['h100_du']))
    prob = rs._SparseQP(np.asarray(args[0]).reshape(-1), *args[1:8])
    lo, hi = rs.qp_bounds(args[2], args[8], args[9], args[10])
    Uk, stats = km.qp_kkt_ipm(prob, lo.T.copy(), hi.T.copy())
    assert Uk is not None and stats['ipm_solves'] <= 25
    assert np.abs(Uk.T - g['h100_U'][i]).max() < 1e-7
