"""CPU tests of the host layer: C-ABI surface, reference-shaped helpers, loud failure without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest

import mpc4quantum_b200 as m4q
from mpc4quantum_b200 import _lib, linearize, systems, vectorize
from mpc4quantum_b200.ensemble import shard_bounds
from oracle import restate as rs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'm4q.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(m4q_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    handle = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared_symbols()
    assert len(names) >= 15
    for name in names:
        assert hasattr(handle, name), name
    assert sorted(_lib.SIGNATURES) == names          # the ctypes table covers exactly the header
    assert _lib.lib().m4q_version() == 100


def test_struct_layout_matches_header():
    assert ctypes.sizeof(_lib.QPSettings) == 48
    # 12 ints, 4 doubles, 8 pointers, the settings, model_per_member + model_mode, noise (2 x 8), streaming +
    # fidelity_sqrt, discount, two stream pointers, member_offset
    assert ctypes.sizeof(_lib.MpcProblem) == 12 * 4 + 4 * 8 + 8 * 8 + 48 + 8 + 16 + 8 + 8 + 16 + 8
    assert _lib.MpcProblem.dt.offset == 48 and _lib.MpcProblem.A_blocks.offset == 80
    assert _lib.MpcProblem.model_per_member.offset == 192 and _lib.MpcProblem.noise_sigma.offset == 200
    assert _lib.MpcProblem.stream_P.offset == 240
    assert lib_sizeof_problem() == ctypes.sizeof(_lib.MpcProblem)


def lib_sizeof_problem():
    """sizeof(m4q_mpc_problem) as the C compiler lays it out (gcc on the header)."""
    import subprocess
    import tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, 's.c')
        with open(src, 'w') as f:
            f.write('#include <stdio.h>\n#include "m4q.h"\nint main(void){printf("%zu", sizeof(m4q_mpc_problem));return 0;}\n')
        exe = os.path.join(tmp, 's')
        subprocess.check_call(['gcc', '-I', os.path.join(root, 'include'), src, '-o', exe])
        return int(subprocess.check_output([exe]))


def test_supported_instantiations_and_argument_errors():
    lib = _lib.lib()
    assert lib.m4q_supported(9, 2) and lib.m4q_supported(4, 1) and lib.m4q_supported(8, 2) and lib.m4q_supported(16, 3)
    assert lib.m4q_supported(16, 1) and lib.m4q_supported(4, 2)
    assert not lib.m4q_supported(5, 1)
    prob = _lib.MpcProblem(c=5, m=1, p=1, d=2, horizon=4, n_steps=2, measure_freq=1, n_targ=7, sat=1.0)
    assert lib.m4q_mpc_table_bytes(ctypes.byref(prob)) == -1
    assert b'unsupported' in lib.m4q_last_error()
    prob = _lib.MpcProblem(c=9, m=2, p=2, d=3, horizon=16, n_steps=20, measure_freq=1, n_targ=37, sat=0.0)
    assert lib.m4q_mpc_state_bytes(ctypes.byref(prob), 4) == -1 and b'sat is mandatory' in lib.m4q_last_error()


def test_launch_geometry_without_a_device():
    lib = _lib.lib()
    prob = _lib.MpcProblem(c=9, m=2, p=2, d=3, horizon=16, n_steps=20, measure_freq=1, n_targ=37, sat=1.0)
    w, c, s = _lib.c_i32(), _lib.c_i32(), _lib.c_i32()
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 0, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert 1 <= w.value <= 16 and c.value % 148 == 0 and s.value <= 227 * 1024
    shared_w, shared_s = w.value, s.value
    prob.model_per_member = 1   # every warp also holds its member's model blocks: 3 * 81 complex more per warp
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 0, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert 1 <= w.value <= shared_w and s.value <= 227 * 1024
    assert (s.value / w.value) - (shared_s / shared_w) > 0.9 * 3 * 81 * 16
    prob.model_per_member = 0
    # few rounds of resident warps (strong scaling): the CTA width is chosen to fill the last round
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 65536, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert w.value == shared_w == 16
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 8192, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert w.value == 14        # 8192 = 3.95 rounds of 148 x 14 instead of 3.46 rounds of 148 x 16
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 100, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert w.value == 1 and c.value == 100      # less than one round of resident warps: spread over the SMs
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 592, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert w.value == 4 and c.value == 148
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 2000, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert w.value == 14 and c.value == 143     # ceil(2000 / 148) warps per CTA, ceil(2000 / 14) CTAs
    prob.horizon = 400          # does not fit the shared-memory slab: refused, not truncated
    assert lib.m4q_mpc_launch_info(ctypes.byref(prob), 0, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == -1
    # c = 16: the slab holds the Riccati scratch P [32][34], G [32][42] and K [m][32]
    gate = _lib.MpcProblem(c=16, m=1, p=1, d=2, horizon=15, n_steps=50, measure_freq=1, lift_mode=_lib.LIFT_PROCESS,
                           n_targ=66, sat=1.0)      # NOT-gate synthesis on process vectors
    assert lib.m4q_mpc_launch_info(ctypes.byref(gate), 0, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert w.value == 8 and c.value == 148      # the MAXW cap of Cfg<16, 1>
    # CNOT state preparation: order-1 model of three controls, p = 3 monomials
    cnot = _lib.MpcProblem(c=16, m=3, p=3, d=4, horizon=50, n_steps=200, measure_freq=1, n_targ=251, sat=1.0)
    assert lib.m4q_mpc_launch_info(ctypes.byref(cnot), 0, ctypes.byref(w), ctypes.byref(c), ctypes.byref(s)) == 0
    assert w.value == 5 and c.value == 148 and s.value <= 227 * 1024


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip('this box has a GPU')
    cfg = systems.config_qubit(1, discretize=rs.taylor_discretize)
    args, kw = systems.mpc_args(cfg)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m4q.mpc(*args, **kw)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m4q.discretize_homogeneous([np.eye(4), np.eye(4)], 1.0, 1)


def test_monomial_tables_match_reference_order():
    assert [list(p) for p in linearize.create_power_list(2, 2)] == rs.power_table(2, 2).tolist()
    assert [list(p) for p in linearize.create_power_list(3, 3)] == rs.power_table(3, 3).tolist()
    assert linearize.size_of_library(2, 2) == 6 and linearize.size_of_library(1, 3) == 4
    u = np.array([[0.5], [-2.0]])
    lib_vals = [f(u)[0] for f in linearize.create_library(2, 2)]
    assert np.allclose(lib_vals, [1, 0.5, 0.25, -2.0, -1.0, 4.0])
    fns, coefs = linearize.diff_library(2, 2)
    d0 = [c[0] * f(u)[0] for f, c in zip(fns[0], coefs[0])]          # d/du1 of u1, u1^2, u2, u1 u2, u2^2
    assert np.allclose(d0, [1, 1.0, 0, -2.0, 0])


def test_krtimes_and_wrapmodel_errors():
    A = np.arange(6.0).reshape(2, 3)
    B = np.arange(12.0).reshape(4, 3)
    K = linearize.krtimes(A, B)
    assert K.shape == (8, 3) and np.allclose(K[:, 1], np.kron(A[:, 1], B[:, 1]))
    with pytest.raises(ValueError):
        linearize.krtimes(A, B[:, :2])
    with pytest.raises(ValueError, match='Dimension mismatch'):
        linearize.WrapModel(np.eye(4), np.zeros((4, 12)), 1, 1)          # linearize.py:23-24


def test_vectorize_me_is_the_liouvillian(unit_golden):
    d = 3
    H = systems.RWA_Transmon(-1.3).H_list[1]
    basis = [np.outer(np.eye(d)[a], np.eye(d)[b]) for a in range(d) for b in range(d)]
    assert np.abs(vectorize.vectorize_me(H, basis) - vectorize.liouvillian(H)).max() < 1e-14
    out = vectorize.vectorize_me(unit_golden['vecme_H'], list(unit_golden['vecme_basis']))
    assert np.abs(out - unit_golden['vecme_out']).max() < 1e-13


def test_stepclock_and_helpers():
    clock = m4q.StepClock(0.25, 16, 20)
    clock.measure_freq = 2
    assert np.allclose(clock.ts, np.linspace(0, 5.0, 20, endpoint=False))
    assert np.allclose(clock.ts_step(3), [0.5, 0.75, 1.0]) and np.allclose(clock.ts_horizon(2)[:2], [0.5, 0.75])
    assert clock.to_string() == 'mf_2d0e00_dt_2d5em01_h_1d6e01_n_2d0e01'
    assert m4q.val_to_str(1.0) == '1d0e00'
    z = np.array([1 + 2j, 3 - 1j])
    assert np.allclose(m4q.real_to_complex(m4q.complex_to_real(z)), z)
    P = np.array([[1 + 1j, 2], [0, 3j]])
    assert np.allclose(m4q.real_to_complex_op(m4q.complex_to_real_op(P)), P)
    assert np.allclose(m4q.shift_guess(np.arange(6.0).reshape(2, 3)), [[1, 2, 2], [4, 5, 5]])
    clock.set_endsim(5)
    assert len(clock.ts_sim) == 5


def test_dmdc_container_and_lifts(unit_golden):
    A = np.arange(24.0).reshape(2, 12)
    model = m4q.DMDc(2, 4, 8, A)
    A_x, A_u = model.get_discrete()
    assert A_x.shape == (2, 4) and A_u.shape == (2, 8)
    assert np.allclose(model.predict(np.ones(4), np.ones(8)), A.sum(axis=1, keepdims=True))
    assert np.abs(m4q.QCoupledExperiment.lift(unit_golden['lift_rho']) - unit_golden['lift_out']).max() < 1e-14
    assert np.abs(m4q.QCoupledExperiment.proj(unit_golden['lift_out']) - unit_golden['proj_out']).max() < 1e-14
    rho3 = np.diag([0.6, 0.3, 0.1]).astype(complex).reshape(-1)
    assert np.allclose(m4q.QExperiment32.lift(rho3), np.diag([2 / 3, 1 / 3]).reshape(-1))
    assert m4q.isqrt(16) == 4
    with pytest.raises(NotImplementedError):
        m4q.DMDc(2, 4, 8, A).fit_iteration(None, None, None)      # read-only container (model.py:70-79)


def test_online_and_discrepancy_dmdc_match_the_reference():
    """model.py:109-313 against vectors produced by the reference's own classes (oracle/make_golden_streaming.py)."""
    from conftest import load_golden
    g = load_golden('streaming')
    dy, dx, du = 4, 4, 8
    mdl = m4q.OnlineDMDc.from_bootstrap(dy, dx, du, g['on_A0'].copy(), alpha=1e2)
    mdl.discount = 0.95
    A_first = mdl.A
    for k in range(6):
        A_x, A_u = mdl.fit_iteration(g['on_y'][k], g['on_x'][k], g['on_u'][k])
    assert np.abs(mdl.A - g['on_A']).max() < 1e-12 and np.abs(mdl.P - g['on_P']).max() < 1e-10
    assert A_x.shape == (dy, dx) and A_u.shape == (dy, du) and np.array_equal(np.hstack([A_x, A_u]), mdl.A)
    assert mdl.A is not A_first and np.array_equal(A_first, g['on_A0'])   # rebinding, not in place (see mpc streaming)
    assert np.abs(mdl.predict(g['on_x'][0], g['on_u'][0]) - g['on_pred']).max() < 1e-12
    mdl = m4q.OnlineDMDc.from_data(g['on_Y'], g['on_X'], g['on_U'])
    mdl.fit_iteration(g['on_y'][0], g['on_x'][0], g['on_u'][0])
    assert np.abs(mdl.A - g['on_data_A']).max() < 1e-10 and np.abs(mdl.P - g['on_data_P']).max() < 1e-10

    mdl = m4q.DiscrepDMDc.from_data(g['on_Y'], g['on_X'], g['on_U'], rcond=1e-8)
    assert np.abs(mdl.A - g['di_A0']).max() < 1e-12
    mdl.discount = 0.9
    for k in range(3):
        mdl.fit_iteration(g['on_y'][k], g['on_x'][k], g['on_u'][k])
    assert np.abs(mdl.A - g['di_A']).max() < 1e-10 and np.abs(mdl.Y - g['di_Ystack']).max() < 1e-13
    mdl = m4q.DiscrepDMDc.from_bootstrap(dy, dx, du, g['on_A0'].copy())
    for k in range(2):
        mdl.fit_iteration(g['on_y'][k], g['on_x'][k], g['on_u'][k])
    assert np.array_equal(mdl.A, g['di_boot_A_rank_deficient']) and np.array_equal(mdl.A, g['on_A0'])   # rank < dim_x
    for k in range(2, 6):
        mdl.fit_iteration(g['on_y'][k], g['on_x'][k], g['on_u'][k])
    assert np.abs(mdl.A - g['di_boot_A']).max() < 1e-9
    mdl._save, mdl._isave = True, 1
    mdl.fit_iteration(g['on_y'][0], g['on_x'][0], g['on_u'][0])
    assert len(mdl.iA) == 2


def test_ensemble_draws_are_reproducible_and_shardable():
    e1, p1 = systems.ensemble_transmon(64)
    e2, p2 = systems.ensemble_transmon(64)
    assert np.array_equal(e1.H0, e2.H0) and e1.H1.shape == (64, 2, 3, 3)
    assert np.allclose(e1.H0, e1.H0.conj().transpose(0, 2, 1))
    bounds = [shard_bounds(65536 + 3, r, 8) for r in range(8)]
    assert bounds[0][0] == 0 and bounds[-1][1] == 65539
    assert all(bounds[i][1] == bounds[i + 1][0] for i in range(7))
    assert max(b - a for a, b in bounds) - min(b - a for a, b in bounds) == 1
    sl = e1.slice(*shard_bounds(64, 1, 4))
    assert len(sl) == 16 and np.array_equal(sl.H0, e1.H0[16:32])


def test_qsynthesis_lift_proj_match_the_reference():
    """QSynthesis.lift / proj (experiment.py:357-388) against vectors from the reference's own statics; QProcess keeps
    them as from_unitary / to_unitary and shows the loop identity maps."""
    from conftest import load_golden
    g = load_golden('gate')
    for n in (2, 3):
        for U, p, b in zip(g['U%d' % n], g['lift%d' % n], g['proj%d' % n]):
            assert np.abs(m4q.QSynthesis.lift(U.reshape(-1)) - p).max() < 1e-15
            assert np.abs(m4q.QSynthesis.proj(p) - b).max() < 1e-14
            assert np.abs(m4q.QProcess.from_unitary(m4q.QProcess.to_unitary(p)) - p).max() < 1e-13
    p = g['lift2'][0]
    assert m4q.QProcess.lift(p) is p and m4q.QProcess.proj(p) is p
    assert m4q.QProcess.lift_mode == 3 and m4q.split_blocks(np.arange(16).reshape(4, 4), 2, 2).shape == (4, 2, 2)


def test_model_containers_for_ensembles_and_exact_mode():
    """Host-side containers added for the ensemble entry point: DMDcEnsemble (perturbed models) and ExactModel."""
    L, params = systems.transmon_model_liouvillians(6)
    assert L.shape == (6, 3, 9, 9) and set(params) == {'model_anharm_scale', 'model_amplitude_scale'}
    for k in range(6):        # batched Liouvillians == the single-model helper (vectorize.py:52-75 in the |a><b| basis)
        a = systems.destroy(3)
        H0 = params['model_anharm_scale'][k] * (-2 * np.pi * 0.1 / 0.25) * systems.proj(3, 2)
        HX = params['model_amplitude_scale'][k] * 0.5 * (a.conj().T + a)
        assert np.abs(L[k, 0] - vectorize.liouvillian(H0)).max() < 1e-15
        assert np.abs(L[k, 1] - vectorize.liouvillian(HX)).max() < 1e-15
    A = np.stack([rs.taylor_discretize(list(L[k]), 0.25, 1) for k in range(6)])
    ens = m4q.DMDcEnsemble(9, 9, 18, A)
    assert len(ens) == 6 and len(ens.slice(2, 5)) == 3
    Ax, Au = ens.member(4).get_discrete()
    assert Ax.shape == (9, 9) and Au.shape == (9, 18) and np.array_equal(np.hstack([Ax, Au]), A[4])
    assert np.array_equal(ens.get_discrete()[0], A[0][:, :9])
    ex = m4q.ExactModel(list(L[0]), 0.25)
    assert (ex.dim_x, ex.dim_u, ex.dt) == (9, 2, 0.25) and ex.generators.shape == (3, 9, 9)
    cfg = systems.config_transmon_exact(horizon=4, n_steps=2)
    assert isinstance(cfg['model'], m4q.ExactModel) and cfg['model'].dim_u == cfg['dim_u']
    gate = systems.config_not_gate(1, discretize=rs.taylor_discretize)
    assert gate['x0'].shape == (16,) and gate['model'].A.shape == (16, 32) and gate['experiment'].lift_mode == 3
    # ||p - pf||^2 = 8 (1 - F): the reference test's callback and the device threshold are the same statement
    p = gate['x0']
    pf = gate['X_targ'][:, 0]
    assert abs(np.vdot(p - pf, p - pf).real - 8 * (1 - np.real(np.vdot(gate['target'], p)))) < 1e-12


def test_shard_draws_equal_slices_of_the_full_draw():
    """Every rank draws only its block of the seeded ensemble (PCG64.advance): bit-identical to slicing the full draw, for
    every ensemble and for ragged shard bounds."""
    from mpc4quantum_b200.ensemble import shard_bounds
    n_total, world = 1001, 3
    for maker in (systems.ensemble_qubit, systems.ensemble_transmon, systems.ensemble_crosstalk, systems.ensemble_not_gate):
        full, params = maker(n_total)
        seen = 0
        for rank in range(world):
            lo, hi = shard_bounds(n_total, rank, world)
            part, pp = maker(n_total, lo=lo, hi=hi)
            assert np.array_equal(part.H0, full.H0[lo:hi]) and np.array_equal(part.H1, full.H1[lo:hi])
            for k in params:
                assert np.array_equal(pp[k], params[k][lo:hi])
            seen += len(part)
        assert seen == n_total
    L, _ = systems.transmon_model_liouvillians(257)
    L2, _ = systems.transmon_model_liouvillians(257, lo=250, hi=257)
    assert np.array_equal(L[250:], L2)
    # the legacy stream: what np.random.default_rng(seed).uniform(.., N) gave before sharding existed
    rng = np.random.default_rng(systems.ENSEMBLE_SEED)
    k = rng.uniform(0.9, 1.1, 64)
    assert np.array_equal(systems.ensemble_transmon(64)[1]['anharm_scale'], k)


def test_kkt_workspaces_are_part_of_the_table_size_only_when_asked_for():
    """m4q_qp_settings.kkt_fallback (include/m4q.h): the pivoted-KKT workspaces, H W (2W + 2) doubles per resident warp
    plus the elimination window and the stored solution (W = 2n + m unknowns per stage), enter m4q_mpc_table_bytes /
    m4q_qp_workspace_bytes_kkt only when the setting is on.  No device needed: the geometry falls back to 148 SMs."""
    lib = _lib.lib()
    c, m, H = 9, 2, 100
    sizes = {}
    for kkt in (0, 2):
        pr = _lib.MpcProblem()
        pr.c, pr.m, pr.p, pr.d, pr.horizon, pr.n_steps, pr.measure_freq = c, m, 2, 3, H, 20, 1
        pr.n_targ, pr.sat = H + 21, 1.0
        pr.qp = _lib.qp_settings(kkt_fallback=kkt)
        sizes[kkt] = int(lib.m4q_mpc_table_bytes(ctypes.byref(pr)))
        w, ctas, smem = _lib.c_i32(), _lib.c_i32(), _lib.c_i32()
        assert lib.m4q_mpc_launch_info(ctypes.byref(pr), 0, ctypes.byref(w), ctypes.byref(ctas), ctypes.byref(smem)) == 0
    assert sizes[0] > 0
    n, W = 2 * c, 4 * c + m
    per_warp = ((W + n) + H * W) * (2 * W + 2) + (H + 2) * W          # Kkt<CF>::doubles(H)
    assert sizes[2] - sizes[0] == 8 * per_warp * w.value * ctas.value
    base = int(lib.m4q_qp_workspace_bytes(4, c, m, H))
    with_kkt = int(lib.m4q_qp_workspace_bytes_kkt(4, c, m, H))
    assert base > 0 and (with_kkt - base) % (8 * per_warp) == 0 and with_kkt > base
    assert _lib.qp_settings().kkt_fallback == 0
