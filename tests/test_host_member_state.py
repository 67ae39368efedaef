"""What a closed-loop member carries between launches, checked without a GPU: the size and layout of the persistent
state, the (shape, order) cases whose streaming model does not fit the slab scratch, and the refusal of measurement
noise on process (gate-synthesis) plants at the Python layer and at the C ABI.

tests/test_gpu_member_state.py runs the launches themselves."""
import ctypes

import numpy as np
import pytest

import mpc4quantum_b200 as m4q
from mpc4quantum_b200 import _lib
from oracle import restate as rs

GRID = [(c, m) for c in (4, 8, 9, 16) for m in (1, 2, 3, 4)]
CASES = [(c, m, order) for c, m in GRID for order in (1, 2) if len(rs.power_table(order, m)) <= 16]
PLANT = {4: (2, _lib.LIFT_IDENTITY), 8: (4, _lib.LIFT_COUPLED), 9: (3, _lib.LIFT_IDENTITY), 16: (4, _lib.LIFT_IDENTITY)}
# MAXBLK + 4 (p + 1) c doubles of z and P z must fit the factor's G buffer, KR LDG doubles (Cfg, m4q_core.cuh)
STREAMING_REFUSED = {(4, 3, 2), (4, 4, 2), (8, 4, 2), (9, 4, 2)}


def _problem(c, m, order, H=16, S=6, **kw):
    d, lift = PLANT[c]
    p = len(rs.power_table(order, m)) - 1
    args = dict(c=c, m=m, p=p, d=d, horizon=H, n_steps=S, measure_freq=1, lift_mode=lift, n_targ=S + H + 1, sat=1.0)
    args.update(kw)
    return _lib.MpcProblem(**args)


def streaming_admitted(c, m, order, H=16):
    """Whether the library plans the fused loop with streaming updates for this case; the refusal must name the
    streaming model."""
    lib = _lib.lib()
    rc = lib.m4q_mpc_launch_info(ctypes.byref(_problem(c, m, order, H, streaming=1)), 0, None, None, None)
    if rc != 0:
        assert b'streaming model too large' in lib.m4q_last_error(), lib.m4q_last_error()
    return rc == 0


def test_streaming_refusals_are_the_cases_whose_model_exceeds_the_scratch():
    lib = _lib.lib()
    refused = set()
    for c, m, order in CASES:
        # without streaming every case plans
        assert lib.m4q_mpc_launch_info(ctypes.byref(_problem(c, m, order)), 0, None, None, None) == 0, (c, m, order)
        if not streaming_admitted(c, m, order):
            refused.add((c, m, order))
    assert refused == STREAMING_REFUSED, sorted(refused)
    # the refusal is about the model size, not the horizon
    for c, m, order in STREAMING_REFUSED:
        assert not streaming_admitted(c, m, order, H=1)


@pytest.mark.parametrize('c,m', GRID)
def test_persistent_state_layout(c, m):
    """Per member: Xg [(H+1) 2c] | Ug, z, y [H m each] | measured plant state [2 max(d^2, c), then as much unused] |
    flags [2].  The prefix keeps the offsets a caller may write the guesses at; the flags word comes last."""
    lib = _lib.lib()
    d, _ = PLANT[c]
    for H in (1, 16, 50):
        for n in (1, 7):
            want = (H + 1) * 2 * c + 3 * H * m + 4 * max(d * d, c) + 2
            assert lib.m4q_mpc_state_bytes(ctypes.byref(_problem(c, m, 1, H)), n) == 8 * n * want, (c, m, H, n)
    # an external (host-stepped) plant carries the lifted model state: d = 0
    ext = _problem(c, m, 1, 16, d=0, lift_mode=_lib.LIFT_IDENTITY)
    assert lib.m4q_mpc_state_bytes(ctypes.byref(ext), 3) == 8 * 3 * (17 * 2 * c + 3 * 16 * m + 4 * c + 2)


def _closed_loop_no_members(prob):
    """m4q_mpc_closed_loop for N = 0: the problem is checked, nothing is launched and no buffer is read."""
    return _lib.lib().m4q_mpc_closed_loop(ctypes.byref(prob), 0, None, 0, None, None, 0, 0, prob.n_steps, 0, None, None,
                                          None, None, None, None, None, None, None, None)


def test_process_plants_refuse_measurement_noise():
    lib = _lib.lib()
    for order in (1, 2):
        process = _problem(16, 2, order, d=2, lift_mode=_lib.LIFT_PROCESS)
        assert _closed_loop_no_members(process) == 0, lib.m4q_last_error()
        process.noise_sigma = 1e-4
        assert _closed_loop_no_members(process) == -1
        assert b'measurement noise is not defined for process' in lib.m4q_last_error()
        # the same noise on a density-matrix plant is accepted
        rho = _problem(16, 2, order, noise_sigma=1e-4)
        assert _closed_loop_no_members(rho) == 0, lib.m4q_last_error()
    H0 = np.zeros((3, 2, 2), complex)
    H1 = np.zeros((3, 2, 2, 2), complex)
    ens = m4q.EnsembleQExperiment(H0, H1, kind='process')
    with pytest.raises(NotImplementedError, match='process'):
        ens.set_sigma(1e-4, seed=1)
    assert ens._sigma == 0.0
    ens.set_sigma(0.0)                        # switching noise off stays allowed
    rho = m4q.EnsembleQExperiment(H0, H1)
    rho.set_sigma(1e-4, seed=1)
    assert rho.slice(1, 2)._sigma == 1e-4
