"""GPU tests of the (dim_x, dim_u) shapes the BASELINE configs leave out (systems.NEW_SHAPES): random QPs, the
linearisation and the closed loop against the restated oracle, and ensembles that must not depend on how their members
are batched."""
import numpy as np
import pytest

import mpc4quantum_b200 as m4q
from mpc4quantum_b200 import optimize, systems
from test_gpu_loop import F_TOL, U_TOL, _exact_oracle, _fid, _oracle_loop
from test_gpu_units import _random_qp

pytestmark = pytest.mark.gpu

SHAPES = systems.NEW_SHAPES


@pytest.mark.parametrize('c,m', SHAPES)
def test_random_qps_match_the_exact_oracle(c, m):
    """Diagonal and full Hermitian costs, with and without the rate bound: the default path and the pivoted KKT solve
    forced on every QP (kkt_fallback = 4) within 1e-8 of the exact solution."""
    from oracle import restate as rs
    rng = np.random.default_rng(3000 * c + m)
    kkt = m4q._lib.qp_settings(kkt_fallback=4)
    for H in (3, 12):
        for hermitian_cost in (False, True):
            for with_du in (True, False):
                a = _random_qp(rng, c, m, H, hermitian_cost, with_du)
                Xc, Uc, objc, info = rs.qp_exact(*a)
                assert max(info['kkt']) < 1e-7
                for settings in (None, kkt):
                    X, U, obj, qinfo = optimize.quad_program(*a, settings=settings)
                    case = (c, m, H, hermitian_cost, with_du, settings is not None)
                    assert qinfo.status_code == 0, case
                    assert np.abs(U - Uc).max() < 1e-8, (case, np.abs(U - Uc).max())
                    assert np.abs(X - Xc).max() < 1e-7, case
                    assert abs(obj - objc) < 1e-8 * max(1.0, abs(objc)), case


@pytest.mark.parametrize('c,m', SHAPES)
def test_linearisation_matches_the_bilinear_model(c, m):
    """WrapModel.get_model_along_traj (device) against restate.BilinearModel at orders 1 and 2 (p + 1 <= 16 blocks)."""
    from oracle import restate as rs
    rng = np.random.default_rng(4000 * c + m)
    H = 7
    for order in (1, 2):
        p1 = len(rs.power_table(order, m))
        A_full = 0.3 * (rng.standard_normal((c, c * p1)) + 1j * rng.standard_normal((c, c * p1))) / np.sqrt(c)
        X = rng.standard_normal((c, H + 1)) + 1j * rng.standard_normal((c, H + 1))
        U = rng.uniform(-1, 1, (m, H))
        A, B, D = m4q.WrapModel(A_full[:, :c], A_full[:, c:], m, order).get_model_along_traj(X, U, np.arange(H))
        Ar, Br, Dr = rs.BilinearModel(A_full, m, order).along(X, U, H)
        for got, ref in ((np.array(A), np.array(Ar)), (np.array(B), np.array(Br)), (np.array(D)[:, :, 0], np.array(Dr))):
            assert got.shape == ref.shape
            assert np.abs(got - ref).max() < 1e-12 * max(1.0, np.abs(ref).max()), (c, m, order)


def _plant_oracle(cfg):
    from oracle import restate as rs
    ex, kind = cfg['experiment'], cfg.get('kind')
    if kind == 'process':
        plant = rs.ProcessPlant(ex.H0, ex.H1_list)
        stats = {}
        xs, us, ec = rs.mpc_loop(cfg['x0'], cfg['dim_u'], cfg['order'], cfg['X_targ'], cfg['U_targ'], cfg['clock'].dt,
                                 cfg['clock'].horizon, cfg['clock'].n_steps, plant, cfg['model'].A, cfg['Q'], cfg['R'],
                                 cfg['Qf'], cfg['sat'], cfg['du'], warm_start=cfg['warm_start'], stats=stats)
        return xs, us, ec, stats
    lift = {None: (None, None), 'coupled': (rs.lift_coupled, rs.proj_coupled), 'trunc32': (rs.lift_32, rs.lift_identity)}
    return _oracle_loop(cfg, ex.H0, ex.H1_list, *lift[kind])


@pytest.mark.parametrize('c,m', SHAPES)
def test_closed_loop_matches_the_restated_loop(c, m):
    """mpc() on each new configuration against restate.mpc_loop with the matching lift: exit codes and per-step SQP
    counts equal, controls within 1e-5, states within 1e-4, final fidelity within 1e-6.  The c = 8 configurations
    measure the plant every second step (model steps in between)."""
    cfg = systems.config_shape(c, m, n_steps=4 if c == 16 else 6)
    if c == 8:
        assert cfg['clock'].measure_freq == 2
    args, kw = systems.mpc_args(cfg)
    (xs, us), _, ec = m4q.mpc(*args, **kw)
    xo, uo, eo, stats = _plant_oracle(cfg)
    assert ec == 0 == eo
    assert np.abs(us - uo).max() < U_TOL, np.abs(us - uo).max()
    assert np.abs(xs - xo).max() < 10 * U_TOL
    assert abs(_fid(cfg, xs[:, -1]) - _fid(cfg, xo[:, -1])) < F_TOL
    # the per-step SQP counts come from a one-member ensemble of the same plant
    ex = cfg['experiment']
    nominal = m4q.EnsembleQExperiment(ex.H0[None], np.stack(ex.H1_list)[None], cfg.get('kind', 'identity'))
    kw.pop('progress_bar')
    res = m4q.mpc_ensemble(args[0], *args[1:6], nominal, *args[7:], **kw)
    assert np.array_equal(res.qp_count[0], stats['qp_per_step']), (res.qp_count[0], stats['qp_per_step'])


@pytest.mark.parametrize('c,m', SHAPES)
def test_ensembles_do_not_depend_on_the_batch(c, m):
    """256 members of ensemble_shape: each member bit for bit equal to a one-member run of its plant, and the same
    members bit for bit equal in two batch compositions (race canary of the warp-private pipeline)."""
    cfg = systems.config_shape(c, m, n_steps=10)
    ens, _ = systems.ensemble_shape(cfg, 256)
    args, kw = systems.mpc_args(cfg)
    kw.pop('progress_bar')

    def run(e):
        return m4q.mpc_ensemble(args[0], *args[1:6], e, *args[7:], fid_target=cfg['target'], **kw)
    a = run(ens)
    b = run(ens.slice(100, 164))
    assert np.array_equal(b.us, a.us[100:164]) and np.array_equal(b.xs, a.xs[100:164])
    assert np.array_equal(b.qp_count, a.qp_count[100:164]) and np.array_equal(b.counters, a.counters[100:164])
    for k in (0, 131, 255):
        s = run(ens.slice(k, k + 1))
        assert np.array_equal(s.us[0], a.us[k]) and np.array_equal(s.xs[0], a.xs[k]), k
        assert np.array_equal(s.exit_code, a.exit_code[k:k + 1]) and np.array_equal(s.qp_count[0], a.qp_count[k])
    assert np.abs(a.us).max() <= cfg['sat'] + 1e-12


def test_host_stepped_equals_fused_on_one_control():
    """(9, 1) through the one-step-per-launch path (a user-defined plant) and through the fused kernel."""
    cfg = systems.config_shape(9, 1, n_steps=6)
    args, kw = systems.mpc_args(cfg)
    (xs_f, us_f), _, ec_f = m4q.mpc(*args, **kw)
    inner = cfg['experiment']

    class MyPlant(m4q.Experiment):
        def f(self, t, x, u):
            raise NotImplementedError

        def simulate(self, x0, ts, us):
            return inner.simulate(x0, ts, us)
    args = list(args)
    args[6] = MyPlant()
    (xs_h, us_h), _, ec_h = m4q.mpc(*args, **kw)
    assert ec_f == ec_h == 0
    assert np.abs(us_h - us_f).max() < 1e-12 and np.abs(xs_h - xs_f).max() < 1e-12


def test_exact_model_on_one_control_matches_oracle():
    """ExactModel (x+ = expm(G(u) dt) x) on the (9, 1) transmon against the restated loop with scipy's expm."""
    from mpc4quantum_b200.vectorize import liouvillian
    cfg = systems.config_shape(9, 1, n_steps=8)
    ex = cfg['experiment']
    cfg['model'] = m4q.ExactModel([liouvillian(h) for h in [ex.H0] + ex.H1_list], cfg['clock'].dt)
    args, kw = systems.mpc_args(cfg)
    (xs, us), _, ec = m4q.mpc(*args, **kw)
    xo, uo, eo, cnt = _exact_oracle(cfg, ex)
    assert ec == 0 == eo
    assert np.abs(us - uo).max() < U_TOL, np.abs(us - uo).max()
    assert np.abs(xs - xo).max() < 10 * U_TOL
    assert abs(_fid(cfg, xs[:, -1]) - _fid(cfg, xo[:, -1])) < F_TOL
