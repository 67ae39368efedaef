"""ctypes binding of libm4q.so (include/m4q.h).  PyTorch is used only to own device memory and streams.

There is no CPU fallback: if the shared library is missing or no CUDA device is present, every compute entry
point raises.  Host-only helpers of the reference API (monomial tables, StepClock, ...) do not come through here.
"""
import ctypes as ct
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('M4Q_LIB') or os.path.join(_HERE, 'libm4q.so')     # M4Q_LIB: measurement aid (build variants)

LIFT_IDENTITY, LIFT_COUPLED, LIFT_TRUNC32, LIFT_PROCESS = 0, 1, 2, 3
MODEL_TAYLOR, MODEL_EXACT = 0, 1

c_i32, c_i64, c_f64, c_vp = ct.c_int32, ct.c_int64, ct.c_double, ct.c_void_p


class QPSettings(ct.Structure):
    """m4q_qp_settings (include/m4q.h)."""
    _fields_ = [('rho', c_f64), ('alpha', c_f64), ('eps', c_f64), ('max_admm', c_i32), ('polish', c_i32),
                ('max_polish', c_i32), ('admm_first', c_i32), ('adaptive_rho', c_i32), ('kkt_fallback', c_i32)]


class MpcProblem(ct.Structure):
    """m4q_mpc_problem (include/m4q.h)."""
    _fields_ = [('c', c_i32), ('m', c_i32), ('p', c_i32), ('d', c_i32), ('horizon', c_i32), ('n_steps', c_i32),
                ('measure_freq', c_i32), ('warm_start', c_i32), ('max_iter', c_i32), ('lift_mode', c_i32),
                ('has_du', c_i32), ('n_targ', c_i32), ('dt', c_f64), ('sat', c_f64), ('du', c_f64),
                ('exit_infidelity', c_f64), ('A_blocks', c_vp), ('powers', c_vp), ('Q', c_vp), ('Qf', c_vp),
                ('R', c_vp), ('X_targ', c_vp), ('U_targ', c_vp), ('fid_vec', c_vp), ('qp', QPSettings),
                ('model_per_member', c_i32), ('model_mode', c_i32), ('noise_sigma', c_f64), ('noise_seed', ct.c_uint64),
                ('streaming', c_i32), ('fidelity_sqrt', c_i32), ('stream_discount', c_f64), ('stream_A', c_vp),
                ('stream_P', c_vp), ('member_offset', c_i64)]


# name -> (restype, argtypes); every symbol include/m4q.h declares
SIGNATURES = {
    'm4q_version': (ct.c_int, []),
    'm4q_last_error': (ct.c_char_p, []),
    'm4q_supported': (ct.c_int, [c_i32, c_i32]),
    'm4q_expm_step_batched': (ct.c_int, [c_i64, c_i32, c_i32, c_i32, c_f64, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp,
                                         c_vp]),
    'm4q_taylor_discretize_batched': (ct.c_int, [c_i64, c_i32, c_i32, c_i32, c_i32, c_f64, c_vp, c_vp, c_vp, c_vp]),
    'm4q_linearize_batched': (ct.c_int, [c_i64, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                         c_vp]),
    'm4q_exact_linearize_batched': (ct.c_int, [c_i64, c_i32, c_i32, c_i32, c_f64] + [c_vp] * 7),
    'm4q_qp_workspace_bytes': (c_i64, [c_i64, c_i32, c_i32, c_i32]),
    'm4q_qp_workspace_bytes_kkt': (c_i64, [c_i64, c_i32, c_i32, c_i32]),
    'm4q_qp_admm_batched': (ct.c_int, [c_i64, c_i32, c_i32, c_i32] + [c_vp] * 9 + [c_f64, c_f64, c_i32,
                                       ct.POINTER(QPSettings)] + [c_vp] * 7),
    'm4q_qp_launch_info': (ct.c_int, [c_i64, c_i32, c_i32, c_i32, ct.POINTER(c_i32), ct.POINTER(c_i32),
                                      ct.POINTER(c_i32)]),
    'm4q_line_search_workspace_bytes': (c_i64, [c_i32, c_i32, c_i32]),
    'm4q_line_search_batched': (ct.c_int, [c_i64, c_i32, c_i32, c_i32] + [c_vp] * 12),
    'm4q_mpc_state_bytes': (c_i64, [ct.POINTER(MpcProblem), c_i64]),
    'm4q_mpc_table_bytes': (c_i64, [ct.POINTER(MpcProblem)]),
    'm4q_mpc_closed_loop': (ct.c_int, [ct.POINTER(MpcProblem), c_i64, c_vp, c_i32, c_vp, c_vp, c_i32, c_i32, c_i32,
                                       c_i32] + [c_vp] * 10),
    'm4q_mpc_herm_sigma': (ct.c_int, [ct.POINTER(MpcProblem), ct.POINTER(c_i32)]),
    'm4q_mpc_factor_counts_offset': (c_i64, [ct.POINTER(MpcProblem)]),
    'm4q_mpc_launch_info': (ct.c_int, [ct.POINTER(MpcProblem), c_i64, ct.POINTER(c_i32), ct.POINTER(c_i32),
                                       ct.POINTER(c_i32)]),
    'm4q_hist_fidelity': (ct.c_int, [c_i64, c_vp, c_f64, c_f64, c_i32, c_vp, c_vp]),
    'm4q_fp64_fma_probe': (ct.c_int, [c_i32, c_i64, c_vp, c_vp]),
    'm4q_fp64_dmma_probe': (ct.c_int, [c_i32, c_i64, c_vp, c_vp]),
}

_lib = None


def lib():
    """The loaded shared library; raises if it has not been built (``python -c 'import __graft_entry__ as g; g.build()'``)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError('libm4q.so is missing at %s: build it with __graft_entry__.build() '
                               '(there is no CPU fallback)' % LIB_PATH)
        handle = ct.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


_shapes = None


def supported_shapes():
    """The (dim_x, dim_u) pairs the library has kernels for, as m4q_supported reports them (every dim_x <= 32 and
    dim_u <= 32 is asked once)."""
    global _shapes
    if _shapes is None:
        handle = lib()
        _shapes = [(c, m) for c in range(1, 33) for m in range(1, 33) if handle.m4q_supported(c, m)]
    return list(_shapes)


def require_shape(c, m):
    """Raise NotImplementedError, naming the compiled pairs, unless (c, m) = (dim_x, dim_u) has kernels."""
    if not lib().m4q_supported(c, m):
        raise NotImplementedError('no compiled kernel for (dim_x, dim_u) = (%d, %d); the compiled pairs are %s'
                                  % (c, m, ', '.join('(%d, %d)' % s for s in supported_shapes())))


def check(rc):
    if rc != 0:
        raise RuntimeError('libm4q: ' + lib().m4q_last_error().decode())


_torch = None


def torch():
    global _torch
    if _torch is None:
        import torch as t
        _torch = t
    return _torch


def require_cuda():
    t = torch()
    if not t.cuda.is_available():
        raise RuntimeError('mpc4quantum_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    lib()
    return t


def dev(x, dtype):
    """Host array (or device tensor) -> contiguous CUDA tensor of the given numpy dtype."""
    t = require_cuda()
    if isinstance(x, t.Tensor):
        want = {np.complex128: t.complex128, np.float64: t.float64, np.int32: t.int32}[dtype]
        return x.to(device='cuda', dtype=want).contiguous()
    return t.from_numpy(np.ascontiguousarray(np.asarray(x), dtype=dtype)).cuda()


def empty(shape, dtype):
    t = require_cuda()
    want = {np.complex128: t.complex128, np.float64: t.float64, np.int32: t.int32, np.int64: t.int64,
            np.uint8: t.uint8}[dtype]
    return t.empty(shape, dtype=want, device='cuda')


def zeros(shape, dtype):
    out = empty(shape, dtype)
    out.zero_()
    return out


def ptr(tensor):
    return c_vp(tensor.data_ptr()) if tensor is not None else c_vp(None)


def stream_ptr(stream=None):
    t = torch()
    st = stream if stream is not None else t.cuda.current_stream()
    return c_vp(st.cuda_stream)


def qp_settings(rho=0.0, alpha=0.0, eps=0.0, max_admm=0, polish=1, max_polish=0, admm_first=0, adaptive_rho=0,
                kkt_fallback=0):
    """Zeros select the library defaults (include/m4q.h)."""
    return QPSettings(rho, alpha, eps, max_admm, polish, max_polish, admm_first, adaptive_rho, kkt_fallback)
