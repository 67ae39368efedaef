"""GPU tests of every compiled (dim_x, dim_u) shape at the edges of its kernels: horizons of one and two stages and
past the KKT-fallback switches, degenerate control boxes, several QP instances per warp, full-width CTAs with a ragged
last one, the exact-model loop on every shape, and the standalone kernels at their size and scaling limits.

References are float64 numpy / scipy (oracle/restate.py), and mpmath at 40 digits where float64 would not be far enough
below the tolerance.  Oracle comparisons are sampled; bit-for-bit comparisons between launches cover the rest."""
import ctypes

import mpmath
import numpy as np
import pytest

import mpc4quantum_b200 as m4q
from mpc4quantum_b200 import _lib, optimize, systems
from mpc4quantum_b200.experiment import expm_segments
from mpc4quantum_b200.mpc import iqp_line_search_batched
from oracle import restate as rs
from test_gpu_loop import F_TOL, U_TOL, _fid
from test_gpu_shapes import _plant_oracle
from test_gpu_units import _random_qp

pytestmark = pytest.mark.gpu

GRID = [(c, m) for c in (4, 8, 9, 16) for m in (1, 2, 3, 4)]
MAXW = {4: 32, 8: 16, 9: 16, 16: 8}     # Tiles<C>::MAXW: warps of a full-width CTA


def _crandn(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


# ----------------------------------------------------------------------------------------------------------
# 1. The QP kernel at short and long horizons and at degenerate control boxes
# ----------------------------------------------------------------------------------------------------------
def _edge_qps(rng, c, m, H):
    """One random QP (test_gpu_units._random_qp) per box edge: (name, arguments of quad_program)."""
    x0, Xb, Ub, Q, R, A, B, D, up, sat, du = _random_qp(rng, c, m, H, False, True)
    sign = np.where(rng.random((m, H)) < 0.5, -1.0, 1.0)
    return [
        # |u_0 - u_prev| <= 0: stage 0 is pinned to u_prev
        ('zero-width stage-0 box', (x0, Xb, Ub, Q, R, A, B, D, np.clip(up, -sat, sat), sat, 0.0)),
        # [-sat, sat] & [u_prev - du, u_prev + du] = {sat}
        ('stage-0 box is the point sat', (x0, Xb, Ub, Q, R, A, B, D, np.full(m, sat + du), sat, du)),
        # targets far outside the box and a control cost that dominates: every control on a bound
        ('every control saturated', (x0, Xb, 3 * sat * sign, Q, [1e6 * r for r in R], A, B, D, sat * sign[:, 0], sat,
                                     du)),
        ('no constraint active', (x0, Xb, Ub, Q, R, A, B, D, up, 1e3, None)),
    ]


@pytest.mark.parametrize('c,m', GRID)
def test_qp_at_horizon_and_box_edges(c, m):
    """H = 1, 2, 5 and 33, 65 (either side of the default kkt_fallback switches at 32 and 64), on the default path and
    with every QP through the pivoted KKT solve (kkt_fallback = 4), against the certified exact oracle."""
    rng = np.random.default_rng(5000 * c + m)
    kkt = _lib.qp_settings(kkt_fallback=4)
    for H in (1, 2, 5, 33, 65):
        for name, a in _edge_qps(rng, c, m, H):
            Xc, Uc, objc, info = rs.qp_exact(*a)
            assert max(info['kkt']) < 1e-7, (name, H, info['kkt'])
            lo, hi = rs.qp_bounds(a[2], a[8], a[9], a[10])
            if name == 'every control saturated':
                assert ((np.abs(Uc - lo) < 1e-12) | (np.abs(Uc - hi) < 1e-12)).all()
            if name == 'no constraint active':
                assert (np.abs(Uc) < 0.5 * a[9]).all()
            for settings in (None, kkt):
                X, U, obj, q = optimize.quad_program(*a, settings=settings)
                case = (c, m, H, name, settings is not None)
                assert q.status_code == 0, case
                err = np.abs(U - Uc).max()
                assert err < (1e-8 if H <= 5 else 1e-6), (case, err)
                assert (U >= lo - 1e-12).all() and (U <= hi + 1e-12).all(), case
                if H <= 5:
                    assert np.abs(X - Xc).max() < 1e-7, case
                else:
                    assert np.abs(X - Xc).max() < 1e-6 * max(1.0, np.abs(Xc).max()), case
                assert abs(obj - objc) < 1e-8 * max(1.0, abs(objc)), (case, obj, objc)


# ----------------------------------------------------------------------------------------------------------
# 2. Several instances per warp in one batched QP launch
# ----------------------------------------------------------------------------------------------------------
def _qp_batch(rng, c, m, H, kinds, sat, du):
    """Random instances of three kinds: 0 mixed, 1 far-out control targets that saturate most controls, 2 an empty
    stage-0 box (u_prev beyond sat + du on one control).  Returns the stacked arguments of quad_program_batched."""
    n = len(kinds)
    rows = []
    for k in range(n):
        x0, Xb, Ub, Q, R, A, B, D, up, _, _ = _random_qp(rng, c, m, H, False, True)
        if kinds[k] == 1:
            Ub = 3 * sat * np.where(rng.random((m, H)) < 0.5, -1.0, 1.0)
        elif kinds[k] == 2:
            up = up.copy()
            up[k % m] = sat + 2 * du
        rows.append((x0, Xb, Ub, np.stack(Q), np.stack(R), np.stack(A), np.stack(B), np.stack(D)[:, :, 0], up))
    return [np.stack(col) for col in zip(*rows)]


def _run_batch(arrays, sat, du, settings, order=None):
    args = [a if order is None else a[order] for a in arrays]
    X, U, obj, status, iters = optimize.quad_program_batched(*args, sat=sat, du=du, settings=settings)
    out = [t.cpu().numpy() for t in (X, U, obj, status, iters)]
    if order is not None:
        inv = np.argsort(order)
        out = [o[inv] for o in out]
    return out


@pytest.mark.parametrize('c,m', GRID)
def test_batched_qp_reuses_slabs_and_kkt_slices(c, m):
    """148 MAXW + 37 instances at H = 8: each warp solves two or more in sequence and the last CTA is ragged.  Every
    instance must equal, bit for bit, the same instance launched in the reversed order (other warps, other
    predecessors), sampled instances must equal one-instance launches, and a leftover working set, mask, counter or KKT
    slice of an infeasible predecessor must not leak into the next instance."""
    H, sat, du = 8, 0.6, 0.25
    n = 148 * MAXW[c] + 37
    w, ctas = _lib.c_i32(), _lib.c_i32()
    _lib.check(_lib.lib().m4q_qp_launch_info(n, c, m, H, ctypes.byref(w), ctypes.byref(ctas), None))
    stride = w.value * ctas.value          # instance k runs on warp k % stride, after instance k - stride
    assert stride < n
    kinds = np.zeros(n, dtype=int)
    kinds[np.arange(n) % 3 == 1] = 1
    kinds[np.arange(n) % 13 == 5] = 2
    after = 5 + stride                     # solved by the warp that has just failed instance 5
    kinds[after] = 0
    feasible = kinds != 2
    rng = np.random.default_rng(6000 * c + m)
    arrays = _qp_batch(rng, c, m, H, kinds, sat, du)
    picks = sorted({0, n - 1, 5, after, int(np.flatnonzero(kinds == 1)[-1]), stride - 1, stride, n // 2})
    oracle = rng.choice(np.flatnonzero(feasible), 20, replace=False)
    certified = {}
    for k in oracle:
        a = [arr[k] for arr in arrays]
        Xc, Uc, objc, info = rs.qp_exact(a[0], a[1], a[2], list(a[3]), list(a[4]), list(a[5]), list(a[6]),
                                         list(a[7][:, :, None]), a[8], sat, du)
        assert max(info['kkt']) < 1e-7, (k, info['kkt'])
        certified[k] = (Xc, Uc, objc)
    for settings in (None, _lib.qp_settings(kkt_fallback=4)):
        X, U, obj, status, iters = _run_batch(arrays, sat, du, settings)
        assert np.array_equal(status == 3, ~feasible), np.flatnonzero((status == 3) != ~feasible)
        assert (status[feasible] == 0).all(), np.flatnonzero(status[feasible] != 0)
        Xr, Ur, objr, statusr, itersr = _run_batch(arrays, sat, du, settings, order=np.arange(n)[::-1])
        assert np.array_equal(statusr, status)
        for got, ref in ((Xr, X), (Ur, U), (objr, obj), (itersr, iters)):
            assert np.array_equal(got[feasible], ref[feasible])
        for k in picks:
            one = _run_batch([arr[k:k + 1] for arr in arrays], sat, du, settings)
            assert one[3][0] == status[k], k
            if feasible[k]:
                for got, ref in zip(one, (X, U, obj, status, iters)):
                    assert np.array_equal(got[0], ref[k]), k
        for k, (Xc, Uc, objc) in certified.items():
            assert np.abs(U[k] - Uc).max() < 1e-8, (k, np.abs(U[k] - Uc).max())
            assert np.abs(X[k] - Xc).max() < 1e-7, k
            assert abs(obj[k] - objc) < 1e-8 * max(1.0, abs(objc)), k


# ----------------------------------------------------------------------------------------------------------
# 3 and 4. The fused loop in full-width CTAs; the exact-model loop on every shape
# ----------------------------------------------------------------------------------------------------------
def _reclock(cfg, horizon=None, n_steps=None):
    """cfg with another horizon / step count, the targets cut or extended to fit."""
    clock = cfg['clock']
    new = m4q.StepClock(dt=clock.dt, horizon=horizon or clock.horizon, n_steps=n_steps or clock.n_steps)
    new.measure_freq = clock.measure_freq
    cols = new.n_steps + new.horizon + 1
    cfg = dict(cfg, clock=new, X_targ=systems._fit_columns(cfg['X_targ'], cols),
               U_targ=systems._fit_columns(cfg['U_targ'], cols - 1))
    return cfg


def _config(c, m, discretize=None):
    """systems.config_shape for the shapes it covers, the BASELINE configuration of the other six."""
    if (c, m) in systems.NEW_SHAPES:
        return systems.config_shape(c, m, discretize=discretize)
    cfg = {(4, 1): lambda: systems.config_qubit(1, discretize=discretize),
           (4, 2): lambda: systems.config_transmon_reduced(discretize=discretize),
           (8, 2): lambda: systems.config_crosstalk(0.05, discretize=discretize),
           (9, 2): lambda: systems.config_transmon(1, discretize=discretize),
           (16, 1): lambda: systems.config_not_gate(1, discretize=discretize),
           (16, 3): lambda: systems.config_cnot(discretize=discretize)}[(c, m)]()
    if (c, m) == (4, 2):
        cfg['target'] = systems.proj(3, 1).reshape(-1)     # fidelity of the plant state, which is a qutrit
    return cfg


def test_fidelity_target_must_match_the_plant_state():
    """The kernel reads one target entry per plant-state entry: a target of the model's size is refused (the reduced
    transmon's model state has 4 entries, its qutrit plant 9)."""
    cfg = systems.config_transmon_reduced(n_steps=2)
    with pytest.raises(ValueError, match='fid_target has 4 entries, the plant state has 9'):
        _run(cfg, _ensemble(cfg, 2))


def _ensemble(cfg, n):
    """n perturbed plants of cfg (systems.ensemble_shape; the BASELINE configs are detuned along diag(0, 1, ...))."""
    d = cfg['experiment'].H0.shape[0]
    cfg = dict(cfg)
    cfg.setdefault('detuning', np.diag(np.arange(d)).astype(complex))
    return systems.ensemble_shape(cfg, n)[0]


def _run(cfg, ens):
    args, kw = systems.mpc_args(cfg)
    kw.pop('progress_bar')
    return m4q.mpc_ensemble(args[0], *args[1:6], ens, *args[7:], fid_target=cfg['target'], **kw)


def _same(a, b, rows=slice(None)):
    for key in ('us', 'xs', 'qp_count', 'counters', 'exit_code', 'steps_done'):
        assert np.array_equal(getattr(a, key)[rows], getattr(b, key)), key


def _full_width_equals_narrow(cfg, c, monkeypatch):
    """3 W + 5 members in CTAs of W warps (M4Q_MAX_WARPS = W switches off the narrowing and tail-aware widths), bit for
    bit equal to the default launch and to one-member runs."""
    n = 3 * MAXW[c] + 5
    ens = _ensemble(cfg, n)
    narrow = _run(cfg, ens)
    with monkeypatch.context() as mp:
        mp.setenv('M4Q_MAX_WARPS', str(MAXW[c]))
        full = _run(cfg, ens)
    _same(full, narrow)
    for k in (0, MAXW[c] - 1, n - 1):
        _same(narrow, _run(cfg, ens.slice(k, k + 1)), slice(k, k + 1))
    return narrow


@pytest.mark.parametrize('c,m', GRID)
def test_fused_loop_in_full_width_ctas(c, m, monkeypatch):
    cfg = _reclock(_config(c, m), n_steps=4 if c == 16 else 6)
    _full_width_equals_narrow(cfg, c, monkeypatch)
    # H = 50, the largest slabs: MAXW copies of the nominal plant in CTAs as wide as they fit, the last copy against the
    # restated loop
    cfg = _reclock(cfg, horizon=50, n_steps=3)
    args, kw = systems.mpc_args(cfg)
    kw.pop('progress_bar')
    ex = cfg['experiment']
    w = MAXW[c]
    nominal = m4q.EnsembleQExperiment(np.repeat(ex.H0[None], w, 0), np.repeat(np.stack(ex.H1_list)[None], w, 0),
                                      cfg.get('kind', 'identity'))
    with monkeypatch.context() as mp:
        mp.setenv('M4Q_MAX_WARPS', str(w))
        res = m4q.mpc_ensemble(args[0], *args[1:6], nominal, *args[7:], **kw)
    xo, uo, eo, _ = _plant_oracle(cfg)
    assert res.exit_code[-1] == eo == 0
    assert np.array_equal(res.us[-1], res.us[0]) and np.array_equal(res.xs[-1], res.xs[0])
    assert np.abs(res.us[-1] - uo).max() < U_TOL, np.abs(res.us[-1] - uo).max()
    xs = res.xs[-1]
    if cfg.get('kind') == 'process':         # the kernel carries the propagator; the oracle the process vector
        xs = np.array([ex.from_unitary(col) for col in xs.T]).T
    assert np.abs(xs - xo).max() < 10 * U_TOL
    assert abs(_fid(cfg, xs[:, -1]) - _fid(cfg, xo[:, -1])) < F_TOL


def _exact_config(c, m):
    """_config with the generators its model was discretised from, as an ExactModel."""
    seen = []

    def capture(L, dt, order):
        seen.append((list(L), dt))
        return rs.taylor_discretize(L, dt, order)
    cfg = _config(c, m, discretize=capture)
    L, dt = seen[-1]                       # the configuration discretises its model last
    assert dt == cfg['clock'].dt and len(L) == m + 1 and L[0].shape == (c, c)
    cfg = _reclock(cfg, horizon=min(cfg['clock'].horizon, 20), n_steps=4)     # scipy's Frechet derivative is the cost
    cfg['model'] = m4q.ExactModel(L, dt)
    cfg['clock'].measure_freq = 1          # the exact model has no model-only steps
    return cfg


def _exact_oracle(cfg, noise=0.0):
    """test_gpu_loop._exact_oracle with the plant of the configuration's lift (test_gpu_shapes._plant_oracle)."""
    ex, kind = cfg['experiment'], cfg.get('kind')

    class Model(rs.ExactModel):
        rng = np.random.default_rng(0)

        def along(self, Xg, Ug, H):
            A, B, D = super().along(Xg, Ug, H)
            if noise:
                A = [a * (1 + noise * self.rng.normal(size=a.shape)) for a in A]
                B = [b * (1 + noise * self.rng.normal(size=b.shape)) for b in B]
                D = [-b @ Ug[:, t] for t, b in enumerate(B)]
            return A, B, D

    if kind == 'process':
        plant = rs.ProcessPlant(ex.H0, ex.H1_list)
    else:
        lift = {None: (rs.lift_identity, rs.lift_identity), 'coupled': (rs.lift_coupled, rs.proj_coupled),
                'trunc32': (rs.lift_32, rs.lift_identity)}[kind]
        plant = rs.ExpmPlant(ex.H0, ex.H1_list, *lift)
    model = Model(list(cfg['model'].generators), cfg['clock'].dt)
    return rs.mpc_loop(cfg['x0'], cfg['dim_u'], cfg['order'], cfg['X_targ'], cfg['U_targ'], cfg['clock'].dt,
                       cfg['clock'].horizon, cfg['clock'].n_steps, plant, None, cfg['Q'], cfg['R'], cfg['Qf'],
                       cfg['sat'], cfg['du'], warm_start=cfg['warm_start'], model=model)


@pytest.mark.parametrize('c,m', GRID)
def test_exact_model_loop_on_every_shape(c, m, monkeypatch):
    """ExactModel built from the configuration's own generators, against the restated loop with scipy's expm and
    expm_frechet.  The tolerance is the north_star's unless this loop amplifies a 1e-15 relative perturbation of A_t and
    B_t -- what any second correctly rounded evaluation amounts to -- by more (test_gpu_loop._exact_oracle).  (4, 3) and
    (4, 4) keep the exact-stage scratch in the record ring's own slab region."""
    cfg = _exact_config(c, m)
    args, kw = systems.mpc_args(cfg)
    (xs, us), _, ec = m4q.mpc(*args, **kw)
    xo, uo, eo = _exact_oracle(cfg)
    assert ec == 0 == eo
    du, df = np.abs(us - uo).max(), abs(_fid(cfg, xs[:, -1]) - _fid(cfg, xo[:, -1]))
    if du >= U_TOL or df >= F_TOL:
        x2, u2, _ = _exact_oracle(cfg, noise=1e-15)
        assert du < max(U_TOL, 20 * np.abs(u2 - uo).max()), du
        assert df < max(F_TOL, 20 * abs(_fid(cfg, x2[:, -1]) - _fid(cfg, xo[:, -1]))), df
    _full_width_equals_narrow(cfg, c, monkeypatch)


# ----------------------------------------------------------------------------------------------------------
# 5. Standalone kernels at their limits
# ----------------------------------------------------------------------------------------------------------
def _line_search_case(rng, c, m, H, n):
    L = _crandn(rng, H + 1, c, c) / np.sqrt(c)
    Q = L @ L.conj().transpose(0, 2, 1)
    Lr = rng.standard_normal((H, m, m))
    R = 0.1 * (Lr @ Lr.transpose(0, 2, 1) + np.eye(m))
    Xr, Ur = _crandn(rng, c, H + 1), rng.standard_normal((m, H))
    Xg, Xo = _crandn(rng, n, c, H + 1), _crandn(rng, n, c, H + 1)
    Ug, Uo = rng.standard_normal((n, m, H)), rng.standard_normal((n, m, H))
    return list(Q), list(R), Xr, Ur, Xg, Ug, Xo, Uo


def _line_search_h_max(c, m):
    """The largest H whose slab and Xg / Xo workspace fit in shared memory, by bisection on the launch's refusal."""
    rng = np.random.default_rng(1)

    def fits(H):
        try:
            iqp_line_search_batched(*_line_search_case(rng, c, m, H, 1))
            return True
        except RuntimeError as e:
            assert 'horizon too long' in str(e)
            return False
    lo, hi = 16, 1024
    assert fits(lo) and not fits(hi)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if fits(mid) else (lo, mid)
    return lo


@pytest.mark.parametrize('c,m', GRID)
def test_line_search_at_short_and_longest_horizons(c, m):
    rng = np.random.default_rng(7000 * c + m)
    for H in (1, 2, 16, _line_search_h_max(c, m)):
        case = _line_search_case(rng, c, m, H, 3)
        alpha, step = (t.cpu().numpy() for t in iqp_line_search_batched(*case))
        Q, R, Xr, Ur, Xg, Ug, Xo, Uo = case
        for k in range(3):
            a, s = rs.line_search(Q, R, Xr, Ur, Xg[k], Ug[k], Xo[k], Uo[k])
            assert abs(alpha[k] - a) < 1e-12 * max(1.0, abs(a)), (H, k, alpha[k], a)
            assert abs(step[k] - s) < 1e-12 * max(1.0, s), (H, k, step[k], s)


def _anti_hermitian(rng, c):
    K = _crandn(rng, c, c)
    return 0.5 * (K - K.conj().T)


def _expm_frechet_mp(G, Es, x):
    """expm(G) and the Frechet derivatives L(G, E) x of an anti-Hermitian G at 40 digits: G = V diag(g) V^H, and
    L(G, E) = V ((V^H E V) o F) V^H with the divided differences F_jk = (e^g_j - e^g_k) / (g_j - g_k) (Daleckii-Krein)."""
    with mpmath.workdps(40):
        lam, V = mpmath.eigh(mpmath.matrix((1j * G).tolist()))     # i G is Hermitian: g = -i lam
        c = G.shape[0]
        g = [-1j * lam[j] for j in range(c)]
        e = [mpmath.exp(gj) for gj in g]
        Vh = V.H
        A = V * mpmath.diag(e) * Vh
        F = mpmath.matrix(c, c)
        for j in range(c):
            for k in range(c):
                dg = g[j] - g[k]
                F[j, k] = e[j] * mpmath.expm1(-dg) / (-dg) if abs(dg) > mpmath.mpf(10) ** -30 else e[j]
        xv = mpmath.matrix(x.tolist())
        bs = []
        for E in Es:
            W = Vh * mpmath.matrix(E.tolist()) * V
            for j in range(c):
                for k in range(c):
                    W[j, k] *= F[j, k]
            bs.append(V * W * (Vh * xv))
        to = lambda M: np.array(M.tolist(), dtype=complex)
        return to(A), np.hstack([to(b) for b in bs])


@pytest.mark.parametrize('c,m', GRID)
def test_exact_linearisation_at_the_scaling_and_substep_switches(c, m):
    """A_t = expm(G dt) and B_t = d/du expm(G dt) x_t with ||G(u) dt||_1 either side of 1/2 (no squaring), 4 (one Taylor
    sub-step of b), 128 and far beyond, for closed-system generators (anti-Hermitian: the exponential stays bounded).
    Above theta = 128 a capped sub-step count truncated the series of b while its partial sums were still large."""
    rng = np.random.default_rng(8000 * c + m)
    # a drift that dominates the 1-norm: ||G dt||_1 is then close to the spectral radius, the size the sub-steps of the
    # Taylor series of b must resolve
    L = [1j * np.diag(rng.uniform(-1, 1, c)) + 0.02 * _anti_hermitian(rng, c) / c]
    L += [0.2 * _anti_hermitian(rng, c) / c for _ in range(m)]
    for theta in (0.49, 0.51, 3.9, 4.1, 127.0, 129.0, 400.0, 1000.0):
        u = rng.uniform(-1, 1, (m, 1))
        G = L[0] + sum(u[i, 0] * L[1 + i] for i in range(m))
        dt = theta / np.abs(G).sum(axis=0).max()
        x = _crandn(rng, c)
        x /= np.linalg.norm(x)
        A, B, D = m4q.ExactModel(L, dt).get_model_along_traj(np.stack([x, x], axis=1), u)
        Ar, Br = _expm_frechet_mp(G * dt, [Li * dt for Li in L[1:]], x)
        tol = 1e-12 * max(1.0, theta)
        assert np.abs(A[0] - Ar).max() < tol, (theta, np.abs(A[0] - Ar).max())
        assert np.abs(B[0] - Br).max() < tol, (theta, np.abs(B[0] - Br).max())
        assert np.abs(D[0][:, 0] + Br @ u[:, 0]).max() < tol


@pytest.mark.parametrize('d', [2, 3, 4])
@pytest.mark.parametrize('m', [3, 4])
def test_plant_expm_with_three_and_four_controls(d, m):
    """expm_segments at N = 4095 (warp per member) and 4096 (thread per member for d <= 4), members whose ||H dt||_1
    sits just below and above 0.5 2^k, against scipy's expm; states against the conjugated reference."""
    from scipy.linalg import expm
    rng = np.random.default_rng(9000 * d + m)
    dt, n_seg = 0.25, 2
    thetas = np.array([0.5 * 2.0 ** k * f for k in range(6) for f in (0.99, 1.01)])
    for n in (4095, 4096):
        K0, K1 = _crandn(rng, n, d, d), _crandn(rng, n, m, d, d)
        H0 = 0.5 * (K0 + K0.conj().transpose(0, 2, 1))
        H1 = 0.5 * (K1 + K1.conj().transpose(0, 1, 3, 2))
        u = rng.uniform(-1, 1, (n, n_seg, m))
        # scale each member's Hamiltonians so that its first segment has the norm thetas[k % len]
        Hu = H0 + np.einsum('ni,nijk->njk', u[:, 0], H1)
        scale = thetas[np.arange(n) % len(thetas)] / (dt * np.abs(Hu).sum(axis=1).max(axis=1))
        H0, H1 = H0 * scale[:, None, None], H1 * scale[:, None, None, None]
        psi = _crandn(rng, n, d)
        psi /= np.linalg.norm(psi, axis=1, keepdims=True)
        rho0 = np.einsum('ni,nj->nij', psi, psi.conj()).reshape(n, d * d)
        states, props = expm_segments(rho0, H0, H1, u, dt, return_propagators=True)
        states, props = states.cpu().numpy(), props.cpu().numpy()
        for k in list(range(2 * len(thetas))) + [n - 2, n - 1]:
            rho = rho0[k].reshape(d, d)
            for sgm in range(n_seg):
                P = expm(-1j * dt * (H0[k] + np.einsum('i,ijk->jk', u[k, sgm], H1[k])))
                assert np.abs(props[k, sgm] - P).max() < 1e-13, (n, k, sgm, np.abs(props[k, sgm] - P).max())
                rho = P @ rho @ P.conj().T
                assert np.abs(states[k, sgm] - rho.reshape(-1)).max() < 1e-12, (n, k, sgm)


@pytest.mark.parametrize('c', [4, 8, 9, 16])
def test_linearisation_at_the_block_limit(c):
    """WrapModel at p + 1 = 16 model blocks (one control at order 15), 15 (two controls at order 4, four at order 2)
    against restate.BilinearModel; 17 blocks (one control at order 16) are refused."""
    rng = np.random.default_rng(10000 + c)
    H = 5
    for m, order in ((1, 15), (2, 4), (4, 2)):
        p1 = len(rs.power_table(order, m))
        assert p1 == (16 if m == 1 else 15)
        A_full = 0.3 * _crandn(rng, c, c * p1) / np.sqrt(c)
        X = _crandn(rng, c, H + 1)
        U = rng.uniform(-1, 1, (m, H))
        A, B, D = m4q.WrapModel(A_full[:, :c], A_full[:, c:], m, order).get_model_along_traj(X, U, np.arange(H))
        Ar, Br, Dr = rs.BilinearModel(A_full, m, order).along(X, U, H)
        for got, ref in ((np.array(A), np.array(Ar)), (np.array(B), np.array(Br)), (np.array(D)[:, :, 0], np.array(Dr))):
            assert np.abs(got - ref).max() < 1e-12 * max(1.0, np.abs(ref).max()), (c, m, order)
    A_full = 0.3 * _crandn(rng, c, c * 17) / np.sqrt(c)
    wm = m4q.WrapModel(A_full[:, :c], A_full[:, c:], 1, 16)
    with pytest.raises(RuntimeError, match='number of monomial blocks out of range'):
        wm.get_model_along_traj(_crandn(rng, c, H + 1), rng.uniform(-1, 1, (1, H)), np.arange(H))
