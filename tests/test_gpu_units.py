"""GPU parity of the individual kernels, through the reference-shaped Python API (which calls the C ABI), against
vectors produced by the reference's own functions (tests/golden/unit.npz, qp.npz; see oracle/make_golden.py)."""
import numpy as np
import pytest

import mpc4quantum_b200 as m4q
from mpc4quantum_b200 import optimize, systems
from mpc4quantum_b200.experiment import expm_segments
from conftest import load_golden

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('tag,orders', [('qubit', (1, 2, 3)), ('transmon', (1, 2, 3)), ('coupled', (1, 2))])
def test_discretize_homogeneous(unit_golden, tag, orders):
    """vectorize.py:8-49; the reference's own test_discretization pins order 1 (tests/test_mpc4quantum.py:182-188)."""
    L = unit_golden['disc_%s_L' % tag]
    dt = float(unit_golden['disc_%s_dt' % tag])
    for o in orders:
        out = m4q.discretize_homogeneous(list(L), dt, o)
        ref = unit_golden['disc_%s_o%d' % (tag, o)]
        assert out.shape == ref.shape
        assert np.abs(out - ref).max() < 1e-13 * max(1.0, np.abs(ref).max())
    c = L.shape[-1]
    o1 = m4q.discretize_homogeneous(list(L), dt, 1)
    assert np.abs(o1 - np.hstack([np.eye(c) + dt * L[0]] + [dt * l for l in L[1:]])).max() < 1e-14


@pytest.mark.parametrize('tag,m', [('qubit', 1), ('transmon', 2), ('transmon1', 2), ('coupled', 3)])
def test_linearize(unit_golden, tag, m):
    """linearize.py:61-70 at random (X, U): A_t, B_t, Delta_t."""
    A_full = unit_golden['lin_%s_A_full' % tag]
    c = A_full.shape[0]
    order = int(unit_golden['lin_%s_order' % tag])
    wm = m4q.WrapModel(A_full[:, :c], A_full[:, c:], m, order)
    X, U = unit_golden['lin_%s_X' % tag], unit_golden['lin_%s_U' % tag]
    H = U.shape[1]
    A, B, D = wm.get_model_along_traj(X, U, np.arange(H))
    for got, ref in ((np.array(A), unit_golden['lin_%s_A' % tag]), (np.array(B), unit_golden['lin_%s_B' % tag]),
                     (np.array(D)[:, :, 0], unit_golden['lin_%s_D' % tag])):
        assert got.shape == ref.shape
        assert np.abs(got - ref).max() < 1e-12 * max(1.0, np.abs(ref).max())
    # single-point entry points agree with the trajectory ones
    assert np.abs(wm.df_dx(X[:, 3], U[:, 3], 0) - A[3]).max() < 1e-13
    assert np.abs(wm.df_du(X[:, 3], U[:, 3], 0) - B[3]).max() < 1e-13
    f = wm.f(X[:, 3], U[:, 3], 0)
    assert np.abs(f[:, 0] - (A[3] @ X[:, 3])).max() < 1e-11 * max(1.0, np.abs(f).max())   # f == A_t x (SURVEY 3.2)


@pytest.mark.parametrize('tag', ['qubit', 'transmon', 'transmon_full', 'cross'])
def test_line_search(unit_golden, tag):
    """mpc.py:101-125 including the time-major / state-major pairing."""
    Q_ls, R_ls = list(unit_golden['ls_%s_Q' % tag]), list(unit_golden['ls_%s_R' % tag])
    X, U = unit_golden['ls_%s_X' % tag], unit_golden['ls_%s_U' % tag]
    alpha, step, _, _ = m4q.iqp_line_search(Q_ls, R_ls, X[0], U[0], X[1], U[1], X[2], U[2])
    assert abs(alpha - float(unit_golden['ls_%s_alpha' % tag])) < 1e-12
    assert abs(step - float(unit_golden['ls_%s_step' % tag])) < 1e-10


@pytest.mark.parametrize('tag,maker', [('qubit', systems.ensemble_qubit), ('transmon', systems.ensemble_transmon),
                                       ('cross', systems.ensemble_crosstalk)])
def test_expm_propagators(unit_golden, tag, maker):
    """Plant propagators within 1e-10 of scipy.linalg.expm (north_star tolerance); conjugation and trace."""
    ens, _ = maker(16)
    u = unit_golden['expm_%s_u' % tag]
    ref = unit_golden['expm_%s_props' % tag]
    dt = float(unit_golden['expm_%s_dt' % tag])
    d = ens.d
    rng = np.random.default_rng(3)
    psi = rng.normal(size=(16, d)) + 1j * rng.normal(size=(16, d))
    psi /= np.linalg.norm(psi, axis=1, keepdims=True)
    rho0 = np.einsum('ni,nj->nij', psi, psi.conj()).reshape(16, d * d)
    states, props = expm_segments(rho0, ens.H0, ens.H1, u, dt, return_propagators=True)
    states, props = states.cpu().numpy(), props.cpu().numpy()
    assert np.abs(props - ref).max() < 1e-10
    assert np.abs(props - ref).max() < 5e-14       # what the kernel actually achieves
    rho = rho0.reshape(16, d, d)
    for sgm in range(3):
        rho = ref[:, sgm] @ rho @ ref[:, sgm].conj().transpose(0, 2, 1)
        assert np.abs(states[:, sgm] - rho.reshape(16, -1)).max() < 1e-12
    assert np.abs(np.einsum('nii->n', states[:, -1].reshape(16, d, d)) - 1).max() < 1e-12


@pytest.mark.parametrize('maker', [systems.ensemble_qubit, systems.ensemble_transmon, systems.ensemble_crosstalk])
@pytest.mark.parametrize('shared', [False, True])
def test_expm_large_ensembles_use_the_thread_per_member_kernel(maker, shared):
    """N >= 4096 and d <= 4 dispatch to the register-resident thread-per-member kernel; it must agree with
    scipy.linalg.expm (north_star 1e-10) and with the warp-per-member kernel (N < 4096) on the same members."""
    from scipy.linalg import expm
    n, n_seg, dt = 8192, 4, 0.25
    ens, _ = maker(n)
    d, m = ens.d, ens.H1.shape[1]
    rng = np.random.default_rng(11)
    u = rng.uniform(-1.5, 1.5, size=(n, n_seg, m))
    psi = rng.normal(size=(n, d)) + 1j * rng.normal(size=(n, d))
    psi /= np.linalg.norm(psi, axis=1, keepdims=True)
    rho0 = np.einsum('ni,nj->nij', psi, psi.conj()).reshape(n, d * d)
    H0, H1 = (ens.H0[5], ens.H1[5]) if shared else (ens.H0, ens.H1)
    big, bigp = expm_segments(rho0, H0, H1, u, dt, shared=shared, return_propagators=True)
    sub = slice(1000, 1064)
    small, smallp = expm_segments(rho0[sub], H0 if shared else H0[sub], H1 if shared else H1[sub], u[sub], dt,
                                  shared=shared, return_propagators=True)
    big, bigp, small, smallp = (t.cpu().numpy() for t in (big, bigp, small, smallp))
    assert np.abs(bigp[sub] - smallp).max() < 1e-13
    assert np.abs(big[sub] - small).max() < 1e-13
    for k in (0, 17, 4095, 4096, n - 1):
        h0, h1 = (H0, H1) if shared else (H0[k], H1[k])
        rho = rho0[k].reshape(d, d)
        for sgm in range(n_seg):
            P = expm(-1j * dt * (h0 + np.einsum('i,ijk->jk', u[k, sgm], h1)))
            assert np.abs(bigp[k, sgm] - P).max() < 1e-13
            rho = P @ rho @ P.conj().T
            assert np.abs(big[k, sgm] - rho.reshape(-1)).max() < 1e-12
    assert np.abs(np.einsum('nii->n', big[:, -1].reshape(n, d, d)) - 1).max() < 1e-12


@pytest.mark.parametrize('tag', ['qubit', 'transmon', 'cross'])
@pytest.mark.parametrize('polish', [1, 0])
def test_quad_program(qp_golden, tag, polish):
    """optimize.py:12-60 against the exact oracle solutions: controls within 1e-8 in the default tight (polished)
    mode -- the mode every parity claim is made in (north_star: 1e-5).  The plain-ADMM mode (polish = 0) stops, like
    OSQP, on residuals; with rho adapted from the residual ratio (m4q_qp_settings.adaptive_rho) it meets the
    north_star's 1e-5 on the controls at eps = 1e-8 within 5,000 iterations (measured, tools/admm_mode_sweep.py:
    1.2e-7 / 2.0e-6 / 3.0e-6 on the qubit / transmon / crosstalk QPs; at eps = 1e-5 and 500 iterations the weakly
    regularised transmon and crosstalk QPs -- R ~ 4e-4 next to B^T P B ~ 1 -- are only 2e-3 / 1e-2 away: a residual of
    1e-5 on these problems is not an error of 1e-5, for OSQP either)."""
    g = qp_golden
    n = g['%s_x_init' % tag].shape[0]
    H = g['%s_U' % tag].shape[2]
    Q_ls = [g['%s_Q' % tag]] * H + [g['%s_Qf' % tag]]
    R_ls = [g['%s_R' % tag]] * H
    settings = m4q._lib.qp_settings(polish=polish, max_admm=5000 if not polish else 0, eps=1e-8 if not polish else 0)
    for i in range(n):
        X, U, obj, info = optimize.quad_program(
            g['%s_x_init' % tag][i], g['%s_X_bm' % tag][i], g['%s_U_bm' % tag][i], Q_ls, R_ls,
            list(g['%s_A' % tag][i]), list(g['%s_B' % tag][i]), list(g['%s_D' % tag][i]), g['%s_u_prev' % tag][i],
            float(g['%s_sat' % tag]), float(g['%s_du' % tag]), settings=settings)
        assert info.status_code == 0
        tol_u = 1e-8 if polish else 1e-5
        assert np.abs(U - g['%s_U' % tag][i]).max() < tol_u, (tag, i, np.abs(U - g['%s_U' % tag][i]).max())
        assert np.abs(X - g['%s_X' % tag][i]).max() < 100 * tol_u
        assert abs(obj - float(g['%s_obj' % tag][i])) < (1e-9 if polish else 1e-6) * max(1.0, abs(float(g['%s_obj' % tag][i])))
        sat, du = float(g['%s_sat' % tag]), float(g['%s_du' % tag])
        assert np.abs(U).max() <= sat + 1e-12
        assert np.abs(U[:, 0] - g['%s_u_prev' % tag][i]).max() <= du + 1e-12


def test_quad_program_h100_order1_pivoted_kkt():
    """QPs of the reference loop at H = 100 with the order-1 model (steps 3, 4, 5, 9: ||prod A_t|| = 1e10 .. 4e13,
    oracle/make_golden_h100.py).  The Riccati path cannot certify them; the pivoted stage-wise KKT solve
    (csrc/m4q_kkt.cuh) must: status 0, controls within 1e-6 of the oracle's sparse solve (itself good to ~1e-8 on the
    worst of them: tools/analysis/abd_full.py compares both with an 80-bit elimination)."""
    g = load_golden('qp_h100')
    n, H = g['h100_U'].shape[0], g['h100_U'].shape[2]
    assert H == 100
    Q_ls = [g['h100_Q']] * H + [g['h100_Qf']]
    R_ls = [g['h100_R']] * H
    sat, du = float(g['h100_sat']), float(g['h100_du'])
    for i in range(n):
        X, U, obj, info = optimize.quad_program(
            g['h100_x_init'][i], g['h100_X_bm'][i], g['h100_U_bm'][i], Q_ls, R_ls, list(g['h100_A'][i]),
            list(g['h100_B'][i]), list(g['h100_D'][i]), g['h100_u_prev'][i], sat, du)
        assert info.status_code == 0, (i, info.status_code)
        err = np.abs(U - g['h100_U'][i]).max()
        assert err < 1e-6, (i, int(g['h100_step'][i]), err)
        assert np.abs(X - g['h100_X'][i]).max() < 1e-6 * max(1.0, np.abs(g['h100_X'][i]).max())
        assert np.abs(U).max() <= sat + 1e-12
        assert np.abs(U[:, 0] - g['h100_u_prev'][i]).max() <= du + 1e-12
    # without the fallback the same problems end with the solver warning (status 2), never with silent garbage
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        X, U, obj, info = optimize.quad_program(
            g['h100_x_init'][0], g['h100_X_bm'][0], g['h100_U_bm'][0], Q_ls, R_ls, list(g['h100_A'][0]),
            list(g['h100_B'][0]), list(g['h100_D'][0]), g['h100_u_prev'][0], sat, du,
            settings=m4q._lib.qp_settings(kkt_fallback=0))
    assert info.status_code in (0, 2)
    if info.status_code == 0:
        assert np.abs(U - g['h100_U'][0]).max() < 1e-5


@pytest.mark.parametrize('c,m', [(4, 1), (4, 2), (9, 2), (8, 2), (16, 3), (16, 1)])
def test_pivoted_kkt_solver_all_instantiations(c, m):
    """The pivoted stage-wise KKT solve + interior-point working set (csrc/m4q_kkt.cuh) forced on every QP
    (kkt_fallback = 4: no Riccati attempt) for every compiled (dim_x, dim_u): random instances with diagonal and full
    Hermitian costs, with and without the rate bound, against the exact oracle -- and against the default
    (Riccati-based) path of the same library.  Block widths 2n + m = 9 .. 67: one to three unknowns per lane."""
    from oracle import restate as rs
    rng = np.random.default_rng(77 * c + m)
    st = m4q._lib.qp_settings(kkt_fallback=4)
    for H in (3, 12):
        for hermitian_cost in (False, True):
            for with_du in (True, False):
                a = _random_qp(rng, c, m, H, hermitian_cost, with_du)
                Xc, Uc, objc, info = rs.qp_exact(*a)
                X, U, obj, qinfo = optimize.quad_program(*a, settings=st)
                assert qinfo.status_code == 0, (c, m, H, hermitian_cost, with_du)
                assert np.abs(U - Uc).max() < 1e-8, (c, m, H, hermitian_cost, with_du, np.abs(U - Uc).max())
                assert np.abs(X - Xc).max() < 1e-7
                assert abs(obj - objc) < 1e-8 * max(1.0, abs(objc))
                X2, U2, obj2, _ = optimize.quad_program(*a)
                assert np.abs(U - U2).max() < 1e-8


def test_quad_program_batched_matches_single(qp_golden):
    g = qp_golden
    tag = 'transmon'
    n, H = g['%s_x_init' % tag].shape[0], g['%s_U' % tag].shape[2]
    Q = np.broadcast_to(np.stack([g['%s_Q' % tag]] * H + [g['%s_Qf' % tag]]), (n, H + 1, 9, 9))
    R = np.broadcast_to(np.stack([g['%s_R' % tag]] * H), (n, H, 2, 2))
    X, U, obj, status, iters = optimize.quad_program_batched(
        g['%s_x_init' % tag], g['%s_X_bm' % tag], g['%s_U_bm' % tag], Q, R, g['%s_A' % tag], g['%s_B' % tag],
        g['%s_D' % tag], g['%s_u_prev' % tag], float(g['%s_sat' % tag]), float(g['%s_du' % tag]))
    assert (status.cpu().numpy() == 0).all()
    assert np.abs(U.cpu().numpy() - g['%s_U' % tag]).max() < 1e-8
    assert (iters.cpu().numpy()[:, 1] >= 2).all()


def test_sat_is_mandatory(qp_golden):
    """optimize.py:43 fails without sat; so do we, loudly."""
    g = qp_golden
    with pytest.raises(TypeError):
        optimize.quad_program(g['qubit_x_init'][0], g['qubit_X_bm'][0], g['qubit_U_bm'][0], [g['qubit_Q']] * 11,
                              [g['qubit_R']] * 10, list(g['qubit_A'][0]), list(g['qubit_B'][0]), list(g['qubit_D'][0]))


def _random_qp(rng, c, m, H, hermitian_cost, with_du):
    """A random instance of the QP of optimize.py:12-60: near-unitary time-varying dynamics, general affine term,
    targets that force part of the controls onto their bounds."""
    def crandn(*shape):
        return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)
    A_ls, B_ls, D_ls = [], [], []
    for _ in range(H):
        K = crandn(c, c)
        A_ls.append(np.eye(c) + 0.15 * (K - K.conj().T) / np.sqrt(c) + 0.01 * crandn(c, c) / np.sqrt(c))
        B_ls.append(0.4 * crandn(c, m))
        D_ls.append(0.05 * crandn(c, 1))
    if hermitian_cost:
        L = crandn(c, c) / np.sqrt(c)
        Q = L @ L.conj().T
        Lf = crandn(c, c) / np.sqrt(c)
        Qf = Lf @ Lf.conj().T
        Lr = rng.standard_normal((m, m))
        R = 0.05 * (Lr @ Lr.T + np.eye(m))
    else:
        Q = np.diag(rng.uniform(0.0, 1.0, c)).astype(complex)
        Qf = 2.0 * Q
        R = np.diag(rng.uniform(0.02, 0.1, m))
    x_init = crandn(c)
    X_bm = crandn(c, H + 1)
    U_bm = 0.3 * rng.standard_normal((m, H))
    sat = 0.6
    du = 0.25 if with_du else None
    # the stage-0 box [-sat, sat] & [u_prev - du, u_prev + du] stays at least du / 2 wide: the QP is feasible
    u_prev = np.clip(0.3 * rng.standard_normal(m), -(sat + 0.125), sat + 0.125)
    return (x_init, X_bm, U_bm, [Q] * H + [Qf], [R] * H, A_ls, B_ls, D_ls, u_prev, sat, du)


@pytest.mark.parametrize('c,m', [(4, 1), (4, 2), (8, 2), (9, 2), (16, 3), (16, 1)])
def test_quad_program_random_instances_all_instantiations(c, m):
    """Every compiled (dim_x, dim_u) kernel against the exact oracle on random QPs: diagonal and full Hermitian costs,
    with and without the rate bound, short and medium horizons.  Tight mode: controls within 1e-8."""
    from oracle import restate as rs
    rng = np.random.default_rng(1000 * c + m)
    worst = 0.0
    for H in (3, 8, 20):
        for hermitian_cost in (False, True):
            for with_du in (True, False):
                a = _random_qp(rng, c, m, H, hermitian_cost, with_du)
                Xc, Uc, objc, info = rs.qp_exact(*a)
                assert max(info['kkt']) < 1e-7
                X, U, obj, qinfo = optimize.quad_program(*a)
                assert qinfo.status_code == 0, (c, m, H, hermitian_cost, with_du)
                err = np.abs(U - Uc).max()
                worst = max(worst, err)
                assert err < 1e-8, (c, m, H, hermitian_cost, with_du, err)
                assert np.abs(X - Xc).max() < 1e-7
                assert abs(obj - objc) < 1e-8 * max(1.0, abs(objc))
                lo, hi = rs.qp_bounds(a[2], a[8], a[9], a[10])
                assert (U >= lo - 1e-12).all() and (U <= hi + 1e-12).all()
                n_active = int((np.abs(Uc - lo) < 1e-9).sum() + (np.abs(Uc - hi) < 1e-9).sum())
                assert 0 <= n_active <= U.size
    assert worst < 1e-8


@pytest.mark.parametrize('tag', ['qubit', 'transmon', 'coupled'])
def test_exact_linearisation_vs_scipy_frechet(unit_golden, tag):
    """Exact-discretisation model mode: A_t = expm(G(u_t) dt) within 1e-10 of scipy.linalg.expm (north_star), and
    B_t = d/du expm(G dt) x_t against scipy.linalg.expm_frechet and a central finite difference."""
    from scipy.linalg import expm
    from oracle import restate as rs
    L = list(unit_golden['disc_%s_L' % tag])
    dt = float(unit_golden['disc_%s_dt' % tag])
    c, m = L[0].shape[0], len(L) - 1
    H = 12
    rng = np.random.default_rng(21)
    X = rng.normal(size=(c, H + 1)) + 1j * rng.normal(size=(c, H + 1))
    U = rng.uniform(-2.0, 2.0, size=(m, H))          # generator norms up to ~6: several sub-steps and squarings
    U[:, 0] = 0.0
    model = m4q.ExactModel(L, dt)
    A, B, D = model.get_model_along_traj(X, U)
    A2, B2, D2 = rs.ExactModel(L, dt).along(X, U, H)
    scale = max(1.0, np.abs(X).max())
    assert np.abs(np.array(A) - np.array(A2)).max() < 1e-12
    assert np.abs(np.array(B) - np.array(B2)).max() < 1e-11 * scale
    assert np.abs(np.array(D)[:, :, 0] - np.array(D2)).max() < 1e-11 * scale * 2
    # independent of scipy's Frechet routine: central difference of expm
    t, eps = 5, 1e-6
    for i in range(m):
        e = np.zeros(m)
        e[i] = eps
        G = lambda u: (L[0] + sum(uk * Lk for uk, Lk in zip(u, L[1:]))) * dt
        fd = (expm(G(U[:, t] + e)) - expm(G(U[:, t] - e))) @ X[:, t] / (2 * eps)
        assert np.abs(B[t][:, i] - fd).max() < 1e-7 * scale
    # consistency with the reference's Taylor model: the order-3 blocks agree with the exact map to O(dt^4)
    if tag == 'qubit':
        return
    A_full = unit_golden['disc_%s_o3' % tag] if ('disc_%s_o3' % tag) in unit_golden else None
    if A_full is not None:
        bm = rs.BilinearModel(A_full, m, 3)
        u_small = 0.1 * U[:, 3]
        A_t = bm.jac_x(u_small)
        A_e = expm((L[0] + sum(uk * Lk for uk, Lk in zip(u_small, L[1:]))) * dt)
        assert np.abs(A_t - A_e).max() < 5e-2
