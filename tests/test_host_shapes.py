"""CPU tests of the compiled (dim_x, dim_u) grid: which pairs exist, their launch geometry without a device, clean
refusals of what does not fit, and the configurations and ensembles of the shapes the BASELINE configs leave out."""
import ctypes

import numpy as np
import pytest

import mpc4quantum_b200 as m4q
from mpc4quantum_b200 import _lib, systems
from oracle import restate as rs

GRID = [(c, m) for c in (4, 8, 9, 16) for m in (1, 2, 3, 4)]
MAXW = {4: 32, 8: 16, 9: 16, 16: 8}
# plant dimension and lift of each state dimension: qubit, two stacked qubits, qutrit, two-qubit density matrix
PLANT = {4: (2, _lib.LIFT_IDENTITY), 8: (4, _lib.LIFT_COUPLED), 9: (3, _lib.LIFT_IDENTITY), 16: (4, _lib.LIFT_IDENTITY)}


def _problem(c, m, order, H, S=20, **kw):
    d, lift = PLANT[c]
    p = len(rs.power_table(order, m)) - 1     # the table's row 0 is the constant monomial
    return _lib.MpcProblem(c=c, m=m, p=p, d=d, horizon=H, n_steps=S, measure_freq=1, lift_mode=lift, n_targ=S + H + 1,
                           sat=1.0, **kw)


def _launch_info(prob, n=0):
    w, ctas, smem = _lib.c_i32(), _lib.c_i32(), _lib.c_i32()
    rc = _lib.lib().m4q_mpc_launch_info(ctypes.byref(prob), n, ctypes.byref(w), ctypes.byref(ctas), ctypes.byref(smem))
    return rc, w.value, ctas.value, smem.value


def test_the_whole_grid_is_compiled():
    lib = _lib.lib()
    for c, m in GRID:
        assert lib.m4q_supported(c, m), (c, m)
    for c, m in ((5, 1), (9, 5), (12, 2)):
        assert not lib.m4q_supported(c, m), (c, m)
    assert m4q.supported_shapes() == GRID


def test_unsupported_shapes_name_the_compiled_ones():
    with pytest.raises(NotImplementedError, match=r'\(5, 1\); the compiled pairs are \(4, 1\), .*\(16, 4\)'):
        _lib.require_shape(5, 1)
    wm = m4q.WrapModel(np.eye(5), np.eye(5), 1, 1)       # the linearisation front end refuses before any device work
    with pytest.raises(NotImplementedError, match=r'\(9, 4\)'):
        wm.get_model_along_traj(np.zeros((5, 4)), np.zeros((1, 3)), np.arange(3))


@pytest.mark.parametrize('c,m', systems.NEW_SHAPES)
def test_launch_geometry_of_the_new_shapes(c, m):
    lib = _lib.lib()
    for order in (1, 2):
        for H in (16, 50):
            prob = _problem(c, m, order, H)
            rc, w, ctas, smem = _launch_info(prob)
            assert rc == 0, (c, m, order, H, lib.m4q_last_error())
            assert 1 <= w <= MAXW[c] and ctas % 148 == 0 and 0 < smem <= 227 * 1024, (c, m, order, H, w, smem)
            assert lib.m4q_mpc_table_bytes(ctypes.byref(prob)) > 0
            assert lib.m4q_mpc_state_bytes(ctypes.byref(prob), 4) > 0
    assert lib.m4q_qp_workspace_bytes(4, c, m, 16) > 0
    assert lib.m4q_qp_workspace_bytes_kkt(4, c, m, 16) >= lib.m4q_qp_workspace_bytes(4, c, m, 16)


def test_shapes_that_do_not_fit_are_refused():
    lib = _lib.lib()
    # three controls at order 3: p = 19 monomials, more blocks than MAXBLK = 16
    prob = _problem(9, 3, 3, 16)
    assert prob.p == 19
    assert _launch_info(prob)[0] == -1 and b'number of monomial blocks out of range' in lib.m4q_last_error()
    prob = _problem(16, 4, 3, 16)
    assert _launch_info(prob)[0] == -1 and b'number of monomial blocks out of range' in lib.m4q_last_error()
    # a horizon whose slab does not fit shared memory
    prob = _problem(16, 4, 2, 400)
    assert _launch_info(prob)[0] == -1 and b'horizon too long' in lib.m4q_last_error()
    # streaming updates of an order-2 model of four controls: 2 x c (p + 1) complex do not fit the c = 4 scratch
    prob = _problem(4, 4, 2, 16, streaming=1)
    assert _launch_info(prob)[0] == -1 and b'streaming model too large' in lib.m4q_last_error()


@pytest.mark.parametrize('c,m', systems.NEW_SHAPES)
def test_configurations_of_the_new_shapes(c, m):
    cfg = systems.config_shape(c, m, n_steps=6, discretize=rs.taylor_discretize)
    assert cfg['dim_u'] == m and cfg['clock'].n_steps == 6
    assert cfg['model'].A.shape == (c, c * (m + 1))
    assert len(cfg['experiment'].H1_list) == m
    assert cfg['R'].shape == (m, m) and cfg['Q'].shape == (c, c)
    assert cfg['X_targ'].shape[1] >= 6 + cfg['clock'].horizon and cfg['U_targ'].shape == (m, 6 + cfg['clock'].horizon)
    d = cfg['experiment'].H0.shape[0]
    assert cfg['detuning'].shape == (d, d)
    if m > 1 and c != 16:
        o2 = systems.config_shape(c, m, order=2, n_steps=6, discretize=rs.taylor_discretize)
        assert o2['model'].A.shape == (c, c * len(rs.power_table(2, m)))


def test_shape_ensemble_shards_equal_slices():
    cfg = systems.config_shape(9, 3, discretize=rs.taylor_discretize)
    full, params = systems.ensemble_shape(cfg, 1000)
    part, pp = systems.ensemble_shape(cfg, 1000, lo=300, hi=420)
    assert np.array_equal(part.H0, full.H0[300:420]) and np.array_equal(part.H1, full.H1[300:420])
    assert np.array_equal(pp['detuning'], params['detuning'][300:420])
    assert full.H1.shape == (1000, 3, 3, 3)
    assert (np.abs(params['amplitude_scale'] - 1) <= 0.1).all()
    assert (np.abs(params['detuning']) <= 0.1 * cfg['sat']).all()
