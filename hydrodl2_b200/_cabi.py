"""ctypes binding of ``include/hbv_b200.h`` (the C-ABI drop-in boundary).

The structures below mirror the header field for field.  There is no CPU
fallback: if the shared library is missing or a call returns non-zero, a
``RuntimeError`` is raised.
"""

from __future__ import annotations

import ctypes as C
import os

HBV_MAX_PAR = 20
HBV_MAX_FLUX = 12
ABI_VERSION = 6

VARIANT_HBV, VARIANT_HBV11P, VARIANT_HBV2, VARIANT_HOURLY, VARIANT_ADJ = 0, 1, 2, 3, 4
SRC_DYN_T, SRC_DYN_LAST, SRC_STA = 0, 1, 2

# flux slots (HBV_F_*)
F_QSIM, F_Q0, F_Q1, F_Q2, F_AET, F_SWE, F_RECHARGE, F_EXCS, F_EVAPFACTOR, F_TOSOIL, F_PERC, \
    F_CAPILLARY = range(12)

_fp = C.c_void_p  # device pointers travel as integers


class HbvDesc(C.Structure):
    _fields_ = [
        ('abi_version', C.c_int32), ('variant', C.c_int32), ('T', C.c_int32), ('B', C.c_int32),
        ('nmul', C.c_int32), ('n_par', C.c_int32), ('betaet', C.c_int32),
        ('apply_sigmoid', C.c_int32), ('nvar', C.c_int32), ('i_prcp', C.c_int32),
        ('i_tmean', C.c_int32), ('i_pet', C.c_int32), ('dyn_ncol', C.c_int32),
        ('sta_ncol', C.c_int32), ('par_src', C.c_int32 * HBV_MAX_PAR),
        ('par_col', C.c_int32 * HBV_MAX_PAR), ('par_lo', C.c_float * HBV_MAX_PAR),
        ('par_hi', C.c_float * HBV_MAX_PAR), ('nearzero', C.c_float), ('dt', C.c_float),
        ('ckpt_interval', C.c_int32), ('muwts_t_stride', C.c_int32), ('adj_max_updates', C.c_int32),
        ('adj_tol', C.c_float), ('ckpt_layout', C.c_int32), ('reserved', C.c_int32 * 3),
    ]


class HbvFwdIO(C.Structure):
    _fields_ = [
        ('forcing', _fp), ('dyn', _fp), ('sta', _fp), ('drop', _fp), ('attrs', _fp),
        ('muwts', _fp), ('state_in', _fp), ('state_out', _fp), ('flux', _fp * HBV_MAX_FLUX),
        ('state_series', _fp), ('ckpt', _fp),
    ]


class HbvBwdIO(C.Structure):
    _fields_ = [
        ('forcing', _fp), ('dyn', _fp), ('sta', _fp), ('drop', _fp), ('attrs', _fp),
        ('muwts', _fp), ('ckpt', _fp), ('gflux', _fp * HBV_MAX_FLUX), ('gstate_out', _fp),
        ('gstate_series', _fp), ('gdyn', _fp), ('gsta', _fp), ('gstate_in', _fp),
        ('gdyn_zero_fill', C.c_int32), ('gdyn_rows_before', C.c_int32), ('gforcing', _fp), ('gmuwts', _fp),
    ]


class HbvTlmIO(C.Structure):
    _fields_ = [
        ('forcing', _fp), ('dyn', _fp), ('sta', _fp), ('drop', _fp), ('attrs', _fp),
        ('muwts', _fp), ('state_in', _fp), ('forcing_t', _fp), ('dyn_t', _fp), ('sta_t', _fp),
        ('muwts_t', _fp), ('state_in_t', _fp), ('flux_t', _fp * HBV_MAX_FLUX), ('state_out_t', _fp),
        ('series_t', _fp), ('flux', _fp * HBV_MAX_FLUX), ('state_out', _fp),
    ]


class HbvAdjFwdIO(C.Structure):
    _fields_ = [
        ('forcing', _fp), ('dyn', _fp), ('drop', _fp), ('state_in', _fp), ('state_out', _fp),
        ('qsim', _fp), ('ysol', _fp), ('stats', _fp),
    ]


class HbvAdjBwdIO(C.Structure):
    _fields_ = [
        ('forcing', _fp), ('dyn', _fp), ('drop', _fp), ('ysol', _fp), ('gqsim', _fp),
        ('gstate_out', _fp), ('gdyn', _fp), ('gstate_in', _fp), ('gdyn_zero_fill', C.c_int32),
        ('gforcing', _fp),
    ]


class HbvRouteDesc(C.Structure):
    _fields_ = [
        ('abi_version', C.c_int32), ('T', C.c_int32), ('B', C.c_int32), ('lenF', C.c_int32),
        ('nser', C.c_int32), ('apply_sigmoid', C.c_int32), ('route_stride', C.c_int32),
        ('bfi_num', C.c_int32), ('bfi_den', C.c_int32), ('a_lo', C.c_float), ('a_hi', C.c_float),
        ('b_lo', C.c_float), ('b_hi', C.c_float), ('nearzero', C.c_float),
        ('reserved', C.c_int32 * 4),
    ]


class HbvPairDesc(C.Structure):
    _fields_ = [
        ('abi_version', C.c_int32), ('T', C.c_int32), ('n_pairs', C.c_int32),
        ('n_units', C.c_int32), ('n_gages', C.c_int32), ('lenF', C.c_int32),
        ('lag_uh', C.c_int32), ('a_lo', C.c_float), ('a_hi', C.c_float), ('b_lo', C.c_float),
        ('b_hi', C.c_float), ('tau_lo', C.c_float), ('tau_hi', C.c_float),
        ('reserved', C.c_int32 * 4),
    ]


EXPORTS = (
    'hbv_b200_fwd', 'hbv_b200_bwd', 'hbv_b200_route_chunks', 'hbv_b200_route_fwd',
    'hbv_b200_route_bwd', 'hbv_b200_abi_version', 'hbv_b200_last_error',
    'hbv_b200_launch_count', 'hbv_b200_pair_chunks', 'hbv_b200_pair_route_fwd',
    'hbv_b200_pair_route_bwd', 'hbv_b200_adj_fwd', 'hbv_b200_adj_bwd', 'hbv_b200_auto_ckpt',
    'hbv_b200_dense_launches', 'hbv_b200_lean_launches', 'hbv_b200_pipe_launches', 'hbv_b200_workspace_bytes',
    'hbv_b200_set_option', 'hbv_b200_get_option', 'hbv_b200_fill_zero', 'hbv_b200_auto_ckpt_desc', 'hbv_b200_copy_cols', 'hbv_b200_memcpy2d', 'hbv_b200_allreduce_buffer_floats', 'hbv_b200_oneshot_allreduce',
    'hbv_b200_tlm', 'hbv_b200_route_tlm',
)

_LIB = None


def lib_path() -> str:
    # HBV_B200_LIB: load an alternative build of the same ABI (e.g. the HBV_MATH=0 precise-math
    # build used by scripts/parity_report.py to quantify the SFU-math error)
    return os.environ.get('HBV_B200_LIB') or os.path.join(
        os.path.dirname(os.path.abspath(__file__)), 'lib', 'libhbv_b200.so')


def load():
    """Load (once) and return the shared library; raise if it is not built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"hydrodl2_b200: CUDA library not found at {path}. Build it with "
            "`python -m hydrodl2_b200._build` (nvcc, sm_100a). There is no CPU fallback."
        )
    lib = C.CDLL(path)
    lib.hbv_b200_abi_version.restype = C.c_int
    if lib.hbv_b200_abi_version() != ABI_VERSION:
        raise RuntimeError('hydrodl2_b200: library ABI version mismatch; rebuild the library')
    lib.hbv_b200_last_error.restype = C.c_char_p
    lib.hbv_b200_launch_count.restype = C.c_int64
    lib.hbv_b200_dense_launches.restype = C.c_int64
    lib.hbv_b200_lean_launches.restype = C.c_int64
    lib.hbv_b200_pipe_launches.restype = C.c_int64
    lib.hbv_b200_workspace_bytes.restype = C.c_int64
    lib.hbv_b200_set_option.restype = C.c_int
    lib.hbv_b200_set_option.argtypes = [C.c_char_p, C.c_int64]
    lib.hbv_b200_get_option.restype = C.c_int64
    lib.hbv_b200_get_option.argtypes = [C.c_char_p]
    lib.hbv_b200_auto_ckpt_desc.restype = C.c_int
    lib.hbv_b200_auto_ckpt_desc.argtypes = [C.POINTER(HbvDesc)]
    lib.hbv_b200_fill_zero.restype = C.c_int
    lib.hbv_b200_fill_zero.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]
    lib.hbv_b200_copy_cols.restype = C.c_int
    lib.hbv_b200_copy_cols.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
    lib.hbv_b200_allreduce_buffer_floats.restype = C.c_int64
    lib.hbv_b200_allreduce_buffer_floats.argtypes = [C.c_int32, C.c_int32]
    lib.hbv_b200_oneshot_allreduce.restype = C.c_int
    lib.hbv_b200_oneshot_allreduce.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.hbv_b200_memcpy2d.restype = C.c_int
    lib.hbv_b200_memcpy2d.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    lib.hbv_b200_workspace_bytes.argtypes = [C.POINTER(HbvDesc)]
    lib.hbv_b200_fwd.restype = C.c_int
    lib.hbv_b200_fwd.argtypes = [C.POINTER(HbvDesc), C.POINTER(HbvFwdIO), C.c_void_p]
    lib.hbv_b200_bwd.restype = C.c_int
    lib.hbv_b200_bwd.argtypes = [C.POINTER(HbvDesc), C.POINTER(HbvBwdIO), C.c_void_p]
    lib.hbv_b200_tlm.restype = C.c_int
    lib.hbv_b200_tlm.argtypes = [C.POINTER(HbvDesc), C.POINTER(HbvTlmIO), C.c_void_p]
    lib.hbv_b200_route_tlm.restype = C.c_int
    lib.hbv_b200_route_tlm.argtypes = [C.POINTER(HbvRouteDesc), _fp, _fp, _fp, C.c_int64, _fp, C.c_int64,
                                       _fp, _fp, _fp, C.c_int64, _fp, _fp, C.c_void_p]
    lib.hbv_b200_adj_fwd.restype = C.c_int
    lib.hbv_b200_adj_fwd.argtypes = [C.POINTER(HbvDesc), C.POINTER(HbvAdjFwdIO), C.c_void_p]
    lib.hbv_b200_adj_bwd.restype = C.c_int
    lib.hbv_b200_adj_bwd.argtypes = [C.POINTER(HbvDesc), C.POINTER(HbvAdjBwdIO), C.c_void_p]
    if hasattr(lib, 'hbv_b200_auto_ckpt'):    # absent only from A/B builds of older sources
        lib.hbv_b200_auto_ckpt.restype = C.c_int
        lib.hbv_b200_auto_ckpt.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    lib.hbv_b200_route_chunks.restype = C.c_int
    lib.hbv_b200_route_chunks.argtypes = [C.c_int32, C.c_int32]
    lib.hbv_b200_route_fwd.restype = C.c_int
    lib.hbv_b200_route_fwd.argtypes = [C.POINTER(HbvRouteDesc), _fp, _fp, C.c_int64, _fp,
                                       C.c_int64, _fp, _fp, _fp, C.c_void_p]
    lib.hbv_b200_route_bwd.restype = C.c_int
    lib.hbv_b200_route_bwd.argtypes = [C.POINTER(HbvRouteDesc), _fp, _fp, C.c_int64, _fp,
                                       C.c_int64, _fp, _fp, _fp, C.c_int64, C.c_uint32, _fp,
                                       _fp, C.c_int64, _fp, _fp, C.c_void_p]
    lib.hbv_b200_pair_chunks.restype = C.c_int
    lib.hbv_b200_pair_chunks.argtypes = [C.c_int32]
    lib.hbv_b200_pair_route_fwd.restype = C.c_int
    lib.hbv_b200_pair_route_fwd.argtypes = [C.POINTER(HbvPairDesc)] + [_fp] * 9 + [C.c_void_p]
    lib.hbv_b200_pair_route_bwd.restype = C.c_int
    lib.hbv_b200_pair_route_bwd.argtypes = [C.POINTER(HbvPairDesc)] + [_fp] * 14 + [C.c_void_p]
    _LIB = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().hbv_b200_last_error().decode(errors='replace')
        kind = 'CUDA error' if rc > 0 else 'argument error'
        raise RuntimeError(f'hydrodl2_b200.{what}: {kind} {rc}: {msg}')


def set_option(name: str, value: int) -> None:
    """Run-time experiment / test switch of the library (include/hbv_b200.h: hbv_b200_set_option);
    value -1 restores the library's own policy."""
    check(load().hbv_b200_set_option(name.encode(), int(value)), f'set_option({name})')


def get_option(name: str) -> int:
    return int(load().hbv_b200_get_option(name.encode()))


class option:
    """Context manager: `with option('lean', 0): ...` sets a switch and restores it on exit."""

    def __init__(self, name: str, value: int):
        self.name, self.value = name, value

    def __enter__(self):
        self.old = get_option(self.name)
        set_option(self.name, self.value)
        return self

    def __exit__(self, *exc):
        set_option(self.name, self.old)
        return False


def launch_count() -> int:
    return int(load().hbv_b200_launch_count())
