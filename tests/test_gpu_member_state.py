"""GPU tests of the state a closed-loop member carries outside one QP, on every compiled (dim_x, dim_u) shape at orders 1
and 2: runs split into step ranges against one launch, the KKT switch across launches, streaming OnlineDMDc updates,
measurement noise on every plant kind, per-member models and the Taylor discretisation kernel they come from.

References are the library's own unsplit launch (bit for bit), host replays of the reference's update rules, the
numpy restatement of the noise generator (test_gpu_stream_noise.py) and float64 numpy / scipy (oracle/restate.py)."""
import numpy as np
import pytest
from scipy.linalg import expm

import mpc4quantum_b200 as m4q
from mpc4quantum_b200 import _lib, systems
from mpc4quantum_b200.linearize import WrapModel, krtimes
from mpc4quantum_b200.mpc import ClosedLoopPlan
from mpc4quantum_b200.vectorize import discretize_homogeneous, discretize_homogeneous_batched
from oracle import restate as rs
from test_gpu_loop import U_TOL
from test_gpu_shape_edges import GRID, MAXW, _config, _ensemble, _plant_oracle, _reclock
from test_gpu_stream_noise import _replay_online_dmdc, normal_pair
from test_host_member_state import CASES, streaming_admitted

pytestmark = pytest.mark.gpu

RESULTS = ('us', 'xs', 'exit_code', 'steps_done', 'qp_count', 'counters', 'fidelity', 'model_A', 'model_P')


def _shape_config(c, m, order):
    """_config of the shape with its model rebuilt at `order` from the generators the configuration discretises (host
    Taylor blocks), horizon at most 20, S = 6 steps (4 for c = 16).  cfg['generators'] holds the generators."""
    seen = []

    def capture(L, dt, o):
        seen.append((list(L), dt))
        return rs.taylor_discretize(L, dt, o)
    cfg = _config(c, m, discretize=capture)
    L, dt = seen[-1]                       # the configuration discretises its model last
    assert dt == cfg['clock'].dt and len(L) == m + 1 and L[0].shape == (c, c)
    cfg = _reclock(cfg, horizon=min(cfg['clock'].horizon, 20), n_steps=4 if c == 16 else 6)
    p1 = len(rs.power_table(order, m))
    cfg.update(order=order, model=m4q.DMDc(c, c, c * (p1 - 1), rs.taylor_discretize(L, dt, order)), generators=L)
    return cfg


def _process(cfg):
    return cfg.get('kind') == 'process'


def _plant_x0(cfg, ens):
    """The configuration's initial plant state as the kernel holds it (the propagator for process plants)."""
    return ens.proj_unitary(cfg['x0']) if _process(cfg) else np.asarray(cfg['x0'], dtype=complex)


def _fidelity(cfg, ens, x):
    """Re<target, x> of a plant state column of xs, as the kernel evaluates it (process: of the lifted propagator)."""
    return float(np.real(np.vdot(cfg['target'], ens.lift_unitary(x) if _process(cfg) else x)))


def _launches(cfg, ens, x0, ranges, exit_infidelity=0.0, model=None, stream=None, settings=None, sigma=0.0, seed=0):
    """One ClosedLoopPlan launched over the step ranges in turn.  Returns the host results after the last launch and
    the factorisation counts summed over the launches."""
    n = len(ens)
    plan = ClosedLoopPlan(cfg['dim_u'], cfg['order'], cfg['X_targ'], cfg['U_targ'], cfg['clock'], model or cfg['model'],
                          cfg['Q'], cfg['R'], cfg['Qf'], cfg['sat'], cfg['du'], ens.d, ens.lift_mode, 100,
                          cfg['warm_start'], cfg['target'], exit_infidelity, settings, n)
    x0d = _lib.dev(x0, np.complex128)
    H0, H1 = _lib.dev(ens.H0, np.complex128), _lib.dev(ens.H1, np.complex128)
    st = None
    if stream is not None:
        A0, P0, disc = stream
        st = (_lib.dev(np.repeat(np.asarray(A0, complex)[None], n, 0), np.complex128),
              _lib.dev(np.repeat(np.asarray(P0, complex)[None], n, 0), np.complex128), disc)
    counts = dict(herm=0, full=0)
    for b, e in ranges:
        res = plan.run(x0d, H0, H1, n=n, step_begin=b, step_end=e, noise_sigma=sigma, noise_seed=seed,
                       member_offset=getattr(ens, 'member_offset', 0), streaming=st)
        for key, v in plan.factor_counts().items():
            counts[key] += v
    return res.numpy(), counts


def _assert_same(got, ref, what):
    for key in RESULTS:
        a, b = getattr(got, key), getattr(ref, key)
        assert (a is None) == (b is None), (what, key)
        if a is not None:
            assert np.array_equal(a, b), (what, key, np.flatnonzero((a != b).reshape(len(a), -1).any(axis=1)))


def _schedules(cfg):
    S = cfg['clock'].n_steps
    out = {'one launch per step': [(s, s + 1) for s in range(S)], 'three launches': [(0, 1), (1, S - 1), (S - 1, S)]}
    if cfg['clock'].measure_freq == 2:
        out['boundary after a model step'] = [(0, 3), (3, S)]      # step 2 is a model step, step 3 a measurement
    return out


def _split_equals_one_launch(cfg, ens, x0, **kw):
    """Every split schedule equals one launch bit for bit, with an exit threshold taken from the unsplit run's own
    states: member 0 (started at the target) stops in step 0, before every split, and at least one member runs to the
    end."""
    S, n = cfg['clock'].n_steps, len(ens)
    free, _ = _launches(cfg, ens, x0, [(0, S)], **kw)
    assert (free.exit_code == 0).all(), free.exit_code
    inf = np.array([[1.0 - _fidelity(cfg, ens, free.xs[k, :, s + 1]) for s in range(S)] for k in range(n)])
    lo, hi = inf[0, 0], inf[1:].min(axis=1).max()
    assert lo < hi, (lo, hi)
    thr = np.sqrt(lo * hi) if lo > 0 else 0.5 * (lo + hi)
    one, counts = _launches(cfg, ens, x0, [(0, S)], exit_infidelity=thr, **kw)
    assert one.exit_code[0] == 1 and one.steps_done[0] == 1, (one.exit_code, one.steps_done)
    assert ((one.exit_code == 0) & (one.steps_done == S)).any(), (one.exit_code, one.steps_done)
    assert counts['herm'] + counts['full'] > 0
    for name, ranges in _schedules(cfg).items():
        split, split_counts = _launches(cfg, ens, x0, ranges, exit_infidelity=thr, **kw)
        _assert_same(split, one, name)
        assert split_counts == counts, (name, split_counts, counts)


def _member_models(cfg, n, order, seed):
    """Per-member generators from the shape's own: drives scaled by U[0.97, 1.03], the drift by U[0.95, 1.05],
    discretised on the device.  Returns the generators [n, m+1, c, c] and the blocks [n, c, c (p+1)]."""
    rng = np.random.default_rng(seed)
    L = np.stack(cfg['generators'])
    drift, drive = rng.uniform(0.95, 1.05, n), rng.uniform(0.97, 1.03, n)
    Ls = np.stack([np.concatenate([drift[k] * L[:1], drive[k] * L[1:]]) for k in range(n)])
    return Ls, discretize_homogeneous_batched(Ls, cfg['clock'].dt, order).cpu().numpy()


def _split_cases():
    return [(c, m, order, variant) for c, m, order in CASES for variant in ('plain', 'streaming', 'model per member')]


# ----------------------------------------------------------------------------------------------------------
# 1. A run split into step ranges equals one launch
# ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('c,m,order,variant', _split_cases())
def test_split_run_equals_one_launch(c, m, order, variant):
    """MAXW + 3 members (one full CTA and a ragged one), noise sigma = 1e-4 except on process plants, members that stop
    at different steps.  Split launches restore each member's guesses, duals, measured state and KKT switch, and leave
    a member that has stopped untouched."""
    cfg = _shape_config(c, m, order)
    if variant == 'streaming' and not streaming_admitted(c, m, order, cfg['clock'].horizon):
        pytest.skip('streaming model too large for the slab scratch (test_host_member_state)')
    n = MAXW[c] + 3
    ens = _ensemble(cfg, n)
    x0 = np.repeat(_plant_x0(cfg, ens)[None], n, 0)
    x0[0] = ens.proj_unitary(4 * cfg['target']) if _process(cfg) else cfg['target']     # starts at the target
    kw = {} if _process(cfg) else dict(sigma=1e-4, seed=0xC0FFEE + 100 * c + 10 * m + order)
    if variant == 'streaming':
        A = cfg['model'].A
        online = m4q.OnlineDMDc.from_bootstrap(c, c, A.shape[1] - c, A.copy(), alpha=10.0)
        kw['stream'] = (online.A, online.P, float(online.discount))
    elif variant == 'model per member':
        _, A = _member_models(cfg, n, order, 100 * c + m)
        kw['model'] = m4q.DMDcEnsemble(c, c, A.shape[2] - c, A)
    _split_equals_one_launch(cfg, ens, x0, **kw)


@pytest.mark.parametrize('c,m', GRID)
def test_a_stopped_member_is_left_untouched(c, m):
    """The empty rate box (test_gpu_stream_noise.test_argument_checks_zeroed_tails_and_the_empty_rate_box): every member
    ends with exit code 3 in step 0.  A second launch from step 3 must not rewrite its steps, fidelity or counters."""
    cfg = _shape_config(c, m, 1)
    cfg['U_targ'] = cfg['U_targ'].copy()
    cfg['U_targ'][:, 0] = 10 * cfg['sat']
    cfg['du'] = 0.1
    ens = _ensemble(cfg, 2)
    x0 = np.repeat(_plant_x0(cfg, ens)[None], 2, 0)
    S = cfg['clock'].n_steps
    first, _ = _launches(cfg, ens, x0, [(0, 3)])
    assert (first.exit_code == 3).all() and (first.steps_done == 0).all()
    assert np.allclose(first.fidelity, [_fidelity(cfg, ens, x) for x in x0], atol=1e-12)
    both, _ = _launches(cfg, ens, x0, [(0, 3), (3, S)])
    _assert_same(both, first, 'second launch')


# ----------------------------------------------------------------------------------------------------------
# 2. The KKT switch of kkt_fallback = 2 across launches
# ----------------------------------------------------------------------------------------------------------
def test_kkt_switch_is_carried_between_launches():
    """Order-1 transmon at H = 100 (default settings: kkt_fallback = 2, the cost-to-go leaves the fp64 range and the
    members switch to the pivoted KKT solve for good): one launch per step equals one launch, counters included."""
    cfg = systems.config_transmon(1, horizon=100, n_steps=8)
    ens, _ = systems.ensemble_transmon(8)
    S = cfg['clock'].n_steps
    x0 = np.repeat(cfg['x0'][None], 8, 0)
    one, counts = _launches(cfg, ens, x0, [(0, S)])
    assert (one.exit_code == 0).all(), one.exit_code
    split, split_counts = _launches(cfg, ens, x0, [(s, s + 1) for s in range(S)])
    _assert_same(split, one, 'one launch per step')
    assert split_counts == counts
    # the premise: the steps before the last split run differently with the KKT solve as the last resort only
    # (kkt_fallback = 1), so mode 2's switch fired in them -- and that switch is what the carried flag holds
    head, _ = _launches(cfg, ens, x0, [(0, S - 1)])
    head1, _ = _launches(cfg, ens, x0, [(0, S - 1)], settings=_lib.qp_settings(kkt_fallback=1))
    assert not np.array_equal(head.counters, head1.counters)


# ----------------------------------------------------------------------------------------------------------
# 3. Streaming OnlineDMDc updates on every shape
# ----------------------------------------------------------------------------------------------------------
class _Wrapped(m4q.Experiment):
    """A user-defined Experiment around a library plant: mpc() steps it on the host, one launch per step."""

    def __init__(self, inner):
        super().__init__()
        self.inner = inner

    def f(self, t, x, u):
        raise NotImplementedError

    def lift(self, x):
        return self.inner.lift(x)

    def proj(self, z):
        return self.inner.proj(z)

    def simulate(self, x0, ts, us):
        return self.inner.simulate(x0, ts, us)


@pytest.mark.parametrize('c,m,order', CASES)
def test_streaming_on_every_shape(c, m, order):
    cfg = _shape_config(c, m, order)
    if not streaming_admitted(c, m, order, cfg['clock'].horizon):
        pytest.skip('streaming model too large for the slab scratch (test_host_member_state)')
    A = cfg['model'].A
    dz = A.shape[1]

    def online():
        return m4q.OnlineDMDc.from_bootstrap(c, c, dz - c, A.copy(), alpha=10.0)
    n = 3
    ens = _ensemble(cfg, n)
    args, kw = systems.mpc_args(cfg)
    kw.pop('progress_bar')
    res = m4q.mpc_ensemble(args[0], *args[1:6], ens, online(), *args[8:], fid_target=cfg['target'], streaming=True,
                           **kw)
    assert (res.exit_code == 0).all(), res.exit_code
    assert np.abs(res.model_A[0] - res.model_A[1]).max() > 1e-9          # every member learns its own plant
    lift = ens.lift_unitary if _process(cfg) else ens.lift
    for k in range(n):
        host = _replay_online_dmdc(online(), cfg, res.xs[k], res.us[k], lift)
        assert np.abs(res.model_A[k] - host.A).max() < 1e-9 * max(1.0, np.abs(host.A).max()), k
        assert np.abs(res.model_P[k] - host.P).max() < 1e-9 * max(1.0, np.abs(host.P).max()), k
        # one member alone through mpc(streaming=True): the same trajectory bit for bit
        member, solo = ens.member(k), online()
        (xs, us), model, ec = m4q.mpc(args[0], *args[1:6], member, solo, *args[8:], streaming=True, progress_bar=False,
                                      **kw)
        want = np.array([member.from_unitary(col) for col in res.xs[k].T]).T if _process(cfg) else res.xs[k]
        assert ec == 0 and np.array_equal(us, res.us[k]) and np.array_equal(xs, want), k
        assert np.array_equal(model.A, res.model_A[k]), k
    # the fused loop against the host-stepped one (the same plant behind a user-defined Experiment)
    fused_model, stepped_model = online(), online()
    (_, us_f), _, ec_f = m4q.mpc(args[0], *args[1:6], ens.member(0), fused_model, *args[8:], streaming=True,
                                 progress_bar=False, **kw)
    (_, us_h), _, ec_h = m4q.mpc(args[0], *args[1:6], _Wrapped(ens.member(0)), stepped_model, *args[8:],
                                 streaming=True, progress_bar=False, **kw)
    assert ec_f == ec_h == 0
    assert np.abs(us_h - us_f).max() < 1e-10, np.abs(us_h - us_f).max()
    scale = max(1.0, np.abs(fused_model.A).max())
    assert np.abs(stepped_model.A - fused_model.A).max() < 1e-10 * scale, np.abs(stepped_model.A - fused_model.A).max()


# ----------------------------------------------------------------------------------------------------------
# 4. Measurement noise on every plant kind
# ----------------------------------------------------------------------------------------------------------
NOISE = {'d = 2': (4, 1), 'd = 3': (9, 4), 'd = 3 trunc32': (4, 2), 'd = 4 coupled': (8, 2), 'd = 4': (16, 3)}


def _conjugate(H0, H1, rho_vec, controls, dt):
    """The plant over consecutive segments, controls[j] on segment j."""
    d = H0.shape[0]
    rho = rho_vec.reshape(d, d)
    for u in controls:
        U = expm(-1j * dt * (H0 + np.einsum('i,ijk->jk', u, H1)))
        rho = U @ rho @ U.conj().T
    return rho.reshape(-1)


@pytest.mark.parametrize('kind', list(NOISE))
def test_measurement_noise_on_every_plant_kind(kind):
    """xs[s + 1] = plant(window) + sigma (n1 + i n2) at every measurement, from the restated generator; model steps
    (measure_freq = 2) carry no noise.  The d = 2 case draws with member_offset = 2^32 + 7, the counter's high word.
    The residuals over the ensemble are N(0, sigma^2) + i N(0, sigma^2), to five standard errors of each moment."""
    c, m = NOISE[kind]
    cfg = _config(c, m)
    cfg = _reclock(cfg, horizon=min(cfg['clock'].horizon, 16), n_steps=10)
    n, sigma, seed = 256, 1e-3, 0x5EED + 10 * c + m
    ens = _ensemble(cfg, n)
    offset = 2 ** 32 + 7 if kind == 'd = 2' else 0
    ens.member_offset = offset
    ens.set_sigma(sigma, seed)
    args, kw = systems.mpc_args(cfg)
    kw.pop('progress_bar')
    res = m4q.mpc_ensemble(args[0], *args[1:6], ens, *args[7:], fid_target=cfg['target'], **kw)
    assert (res.exit_code == 0).all()
    S, mf, dt, d = cfg['clock'].n_steps, cfg['clock'].measure_freq, cfg['clock'].dt, ens.d
    H0, H1 = np.asarray(ens.H0), np.asarray(ens.H1)
    A = cfg['model'].A
    wrapped = WrapModel(A[:, :c], A[:, c:], m, cfg['order'])
    lift, proj = (rs.lift_coupled, rs.proj_coupled) if cfg.get('kind') == 'coupled' else (None, None)
    resid = []
    for k in range(n):
        xs, us = res.xs[k], res.us[k]
        for s in range(S):
            if (s + 1) % mf == 0:
                # the plant from the last measured (noisy) state, newest control first (mpc.py:257)
                plant = _conjugate(H0[k], H1[k], xs[:, s + 1 - mf], [us[:, s - j] for j in range(mf)], dt)
                r = xs[:, s + 1] - plant
                resid.append(r)
                if k in (0, 1, n - 1):
                    want = sigma * np.array([complex(*normal_pair(seed, offset + k, s, comp)) for comp in range(d * d)])
                    assert np.abs(r - want).max() < 1e-12, (k, s, np.abs(r - want).max())
            elif k in (0, 1, n - 1):
                lx = np.asarray(lift(xs[:, s])).reshape(-1, 1)
                lu = wrapped.lift_u(us[:, s].reshape(-1, 1))
                pred = proj((A[:, :c] @ lx + A[:, c:] @ krtimes(lu, lx)).reshape(-1))
                assert np.abs(xs[:, s + 1] - pred).max() < 1e-12, (k, s)
    resid = np.array(resid)
    z = np.concatenate([resid.real.ravel(), resid.imag.ravel()]) / sigma
    ns = len(z)
    assert abs(z.mean()) < 5 / np.sqrt(ns), z.mean()
    assert abs(z.var() - 1) < 5 * np.sqrt(2 / ns), z.var()
    assert abs(np.mean(z ** 3)) < 5 * np.sqrt(15 / ns), np.mean(z ** 3)
    assert abs(np.mean(z ** 4) - 3) < 5 * np.sqrt(96 / ns), np.mean(z ** 4)
    assert abs(np.corrcoef(resid.real.ravel(), resid.imag.ravel())[0, 1]) < 5 / np.sqrt(ns / 2)


def test_process_ensembles_refuse_measurement_noise():
    """The process lift measures a propagator; the reference defines no noise for it.  Refused by
    EnsembleQExperiment.set_sigma and, for a caller of ClosedLoopPlan.run, by m4q_mpc_closed_loop."""
    cfg = _shape_config(16, 2, 1)
    ens = _ensemble(cfg, 2)
    with pytest.raises(NotImplementedError, match='process'):
        ens.set_sigma(1e-4, seed=1)
    x0 = np.repeat(_plant_x0(cfg, ens)[None], 2, 0)
    with pytest.raises(RuntimeError, match='measurement noise is not defined for process'):
        _launches(cfg, ens, x0, [(0, cfg['clock'].n_steps)], sigma=1e-4, seed=1)
    clean, _ = _launches(cfg, ens, x0, [(0, cfg['clock'].n_steps)])
    assert (clean.exit_code == 0).all()


# ----------------------------------------------------------------------------------------------------------
# 5. Per-member models and the Taylor discretisation kernel
# ----------------------------------------------------------------------------------------------------------
def _assert_blocks_close(got, ref, c, what):
    """Each c x c block within 1e-13 of its largest entry (blocks that vanish in the reference: of the whole model's)."""
    top = np.abs(ref).max()
    for b in range(ref.shape[1] // c):
        g, r = got[:, b * c:(b + 1) * c], ref[:, b * c:(b + 1) * c]
        scale = max(np.abs(r).max(), 1e-12 * top)
        assert np.abs(g - r).max() <= 1e-13 * scale, (what, b, np.abs(g - r).max(), scale)


@pytest.mark.parametrize('c,m,order', CASES)
def test_per_member_models(c, m, order):
    """(a) the device discretisation of every member's generators against rs.taylor_discretize; (b) member k of the
    ensemble bit for bit equal to a one-member run of the shared-model path with DMDc(A_k), which for c = 8 and 16 reads
    the transposed block copies; (c) one member against the restated loop with its own model."""
    cfg = _shape_config(c, m, order)
    n = 4
    Ls, A = _member_models(cfg, n, order, 200 * c + m)
    for k in range(n):
        _assert_blocks_close(A[k], rs.taylor_discretize(list(Ls[k]), cfg['clock'].dt, order), c, k)
    ens = _ensemble(cfg, n)
    args, kw = systems.mpc_args(cfg)
    kw.pop('progress_bar')
    p = A.shape[2] // c - 1
    res = m4q.mpc_ensemble(args[0], *args[1:6], ens, m4q.DMDcEnsemble(c, c, c * p, A), *args[8:],
                           fid_target=cfg['target'], **kw)
    assert (res.exit_code == 0).all(), res.exit_code
    for k in (0, n - 1):
        one = m4q.mpc_ensemble(args[0], *args[1:6], ens.slice(k, k + 1), m4q.DMDc(c, c, c * p, A[k]), *args[8:],
                               fid_target=cfg['target'], **kw)
        for key in ('us', 'xs', 'exit_code', 'steps_done', 'qp_count', 'counters', 'fidelity'):
            assert np.array_equal(getattr(one, key)[0], getattr(res, key)[k]), (k, key)
    k = 1
    xo, uo, eo, _ = _plant_oracle(dict(cfg, experiment=ens.member(k), model=m4q.DMDc(c, c, c * p, A[k])))
    assert eo == 0
    assert np.abs(res.us[k] - uo).max() < U_TOL, np.abs(res.us[k] - uo).max()
    if not _process(cfg):
        assert np.abs(res.xs[k] - xo).max() < 10 * U_TOL


# the first order whose blocks do not fit the discretisation kernel's shared memory, 3 p1 c^2 16 + 4 p1 (m + 1) bytes
TAYLOR_REFUSED = {(16, 1): 18, (16, 2): 5, (16, 3): 3, (16, 4): 3}


def _taylor_bytes(c, m, order):
    p1 = len(rs.power_table(order, m))
    return 3 * p1 * c * c * 16 + 4 * p1 * (m + 1)


@pytest.mark.parametrize('c,m', GRID)
def test_taylor_kernel_on_every_shape(c, m):
    """discretize_homogeneous (m4q_taylor_discretize_batched) against rs.taylor_discretize at orders 1 to 3 where the
    kernel's shared memory admits them, order 4 on (16, 2), and the refusal of the first order that does not fit."""
    cfg = _shape_config(c, m, 1)
    L, dt = cfg['generators'], cfg['clock'].dt
    orders = [1, 2, 3] + ([4] if (c, m) == (16, 2) else [])
    for order in orders:
        if _taylor_bytes(c, m, order) > 227 * 1024:
            assert order >= TAYLOR_REFUSED[(c, m)]
            continue
        _assert_blocks_close(discretize_homogeneous(L, dt, order), rs.taylor_discretize(L, dt, order), c, order)
    first = TAYLOR_REFUSED.get((c, m))
    if first is not None:
        assert _taylor_bytes(c, m, first - 1) <= 227 * 1024 < _taylor_bytes(c, m, first)
        with pytest.raises(RuntimeError, match='model too large for the shared-memory discretisation kernel'):
            discretize_homogeneous(L, dt, first)
