"""Launch geometry of every compiled (dim_x, dim_u) shape: the longest horizon each fits, and resident warps that never
outnumber the per-warp workspaces.

The fused loop's tables (m4q_mpc_table_bytes) and the standalone QP's KKT slices (m4q_qp_workspace_bytes_kkt) hold one
workspace per resident warp of the widest launch, the one planned for 2^40 members.  A warp finds its slice at
(blockIdx.x * warps + warp), so a launch for fewer members must never run more warps than that.  Without a device the
planner counts residency from shared memory alone; under the gpu marker the same checks run with the real occupancy
calculator.
"""
import ctypes

import pytest

from mpc4quantum_b200 import _lib
from oracle import restate as rs

GRID = [(c, m) for c in (4, 8, 9, 16) for m in (1, 2, 3, 4)]
PLANT = {4: (2, _lib.LIFT_IDENTITY), 8: (4, _lib.LIFT_COUPLED), 9: (3, _lib.LIFT_IDENTITY), 16: (4, _lib.LIFT_IDENTITY)}
H_CEIL = 1 << 14          # refused by every shape: the slab grows linearly with H
CASES = [(c, m, order) for c, m in GRID for order in (1, 2) if len(rs.power_table(order, m)) <= 16]


def _mpc_info(c, m, order, H, n):
    d, lift = PLANT[c]
    p = len(rs.power_table(order, m)) - 1
    prob = _lib.MpcProblem(c=c, m=m, p=p, d=d, horizon=H, n_steps=20, measure_freq=1, lift_mode=lift, n_targ=21 + H,
                           sat=1.0)
    w, ctas, smem = _lib.c_i32(), _lib.c_i32(), _lib.c_i32()
    rc = _lib.lib().m4q_mpc_launch_info(ctypes.byref(prob), n, ctypes.byref(w), ctypes.byref(ctas), ctypes.byref(smem))
    return rc, w.value, ctas.value, smem.value


def _qp_info(c, m, H, n):
    w, ctas, smem = _lib.c_i32(), _lib.c_i32(), _lib.c_i32()
    rc = _lib.lib().m4q_qp_launch_info(n, c, m, H, ctypes.byref(w), ctypes.byref(ctas), ctypes.byref(smem))
    return rc, w.value, ctas.value, smem.value


def _h_max(info):
    """Largest H that info(H, n) plans, by bisection; H + 1 must be refused as too long for the slab."""
    assert info(1, 0)[0] == 0, _lib.lib().m4q_last_error()
    assert info(H_CEIL, 0)[0] == -1
    lo, hi = 1, H_CEIL
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if info(mid, 0)[0] == 0:
            lo = mid
        else:
            hi = mid
    assert info(lo + 1, 0)[0] == -1 and b'horizon too long' in _lib.lib().m4q_last_error()
    return lo


def _sms():
    """The SM count the planner sees: the device's when there is one, else its no-device default of 148."""
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count if torch.cuda.is_available() else 148


def _member_counts(sms, full, widest):
    """1 .. 8 full waves + 1.  Between two round boundaries k * SMs * w of some width w <= widest the planner's choice
    is fixed and its resident warps grow with N, so the largest counts sit just below, at and just above those
    boundaries; a coarse sweep covers the rest."""
    ns = {1, 8 * full, 8 * full + 1}
    for w in range(1, widest + 1):
        for k in range(1, 9):
            ns.update(k * sms * w + d for d in (-1, 0, 1))
    ns.update(range(1, 8 * full + 2, max(1, full // 97)))
    return sorted(n for n in ns if 1 <= n <= 8 * full + 1)


def _check_residency(info, H, sms):
    rc, w0, c0, smem0 = info(H, 0)
    assert rc == 0, _lib.lib().m4q_last_error()
    assert 1 <= w0 and 1 <= c0 and 0 < smem0 <= 227 * 1024
    cap = w0 * c0
    for n in _member_counts(sms, sms * w0, w0):
        rc, w, ctas, smem = info(H, n)
        assert rc == 0, (n, _lib.lib().m4q_last_error())
        assert w * ctas <= cap, ('H', H, 'N', n, 'warps', w, 'ctas', ctas, 'the tables hold', cap)
        assert 1 <= w <= w0 and 1 <= ctas and smem <= smem0


def _horizons(h_max):
    return sorted(h for h in {1, 2, 16, 50, h_max} if h <= h_max)


def _mpc_case(c, m, order, sms):
    def info(H, n):
        return _mpc_info(c, m, order, H, n)
    h_max = _h_max(info)
    for H in _horizons(h_max):
        _check_residency(info, H, sms)
    return h_max


def _qp_case(c, m, sms):
    def info(H, n):
        return _qp_info(c, m, H, n)
    h_max = _h_max(info)
    for H in _horizons(h_max):
        _check_residency(info, H, sms)
    return h_max


@pytest.mark.parametrize('c,m,order', CASES)
def test_fused_loop_never_runs_more_warps_than_its_tables_hold(c, m, order):
    h_max = _mpc_case(c, m, order, _sms())
    assert h_max >= 50, h_max


@pytest.mark.parametrize('c,m', GRID)
def test_standalone_qp_never_runs_more_warps_than_its_kkt_slices(c, m):
    h_max = _qp_case(c, m, _sms())
    assert h_max >= 100, h_max
    assert _lib.lib().m4q_qp_workspace_bytes_kkt(1, c, m, h_max) > _lib.lib().m4q_qp_workspace_bytes(1, c, m, h_max)


def test_tail_aware_width_keeps_one_cta_per_sm():
    """Two cases where the narrower tail-aware width would fit two CTAs per SM without a device: one full wave + 1
    members of (8, 1) at H = 16, and four waves + 1 of (4, 4) at H = 1."""
    for (c, m, H), waves in (((8, 1, 16), 1), ((4, 4, 1), 4)):
        rc, w0, c0, _ = _mpc_info(c, m, 1, H, 0)
        assert rc == 0
        rc, w, ctas, _ = _mpc_info(c, m, 1, H, waves * c0 * w0 + 1)
        assert rc == 0 and w * ctas <= w0 * c0, (c, m, H, w0, c0, w, ctas)


def test_qp_launch_info_refusals():
    lib = _lib.lib()
    assert _qp_info(5, 1, 8, 0)[0] == -1 and b'unsupported (c, m)' in lib.m4q_last_error()
    assert _qp_info(9, 2, 0, 0)[0] == -1 and b'horizon out of range' in lib.m4q_last_error()
    rc, w, ctas, smem = _qp_info(9, 2, 16, 5)
    assert rc == 0 and w == 1 and ctas == 5


@pytest.mark.gpu
@pytest.mark.parametrize('c,m', GRID)
def test_residency_with_the_occupancy_calculator(c, m):
    """The checks above with the device's SM count, shared memory and register-limited occupancy."""
    _lib.require_cuda()
    for order in (1, 2):
        if (c, m, order) in CASES:
            _mpc_case(c, m, order, _sms())
    _qp_case(c, m, _sms())
