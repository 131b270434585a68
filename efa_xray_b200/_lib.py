"""ctypes binding of include/efa_xray_b200.h.

The library is the product: there is no CPU or PyTorch fallback.  If the shared object has not been
built, or no sm_100 device is present, the calls raise.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libefa_xray_b200.so')

_p = C.c_void_p
_i64 = C.c_int64
_int = C.c_int
_dbl = C.c_double

# name -> argtypes; every function returns int status except exb_last_error
SIGNATURES = {
    'exb_version': [],
    'exb_device_check': [],
    'exb_grid_unitvec': [_p, _p, _i64, _p, _p],
    'exb_obs_trig': [_p, _p, _i64, _p, _p, _p],
    'exb_obs_prepare': [_p, _p, _p, _i64, _int, _p, _p],
    'exb_stencil_search': [_p, _p, _p, _p, _i64, _p, _p, _p, _p, _i64, _p, _p, _p, _p],
    'exb_stencil_search_rect': [_p, _p, _p, _p, _i64, _i64, _p, _p, _p, _p, _i64, _p, _p, _p, _p],
    'exb_pseudo_distance': [_p, _p, _i64, _dbl, _dbl, _p, _p],
    'exb_stencil_bilinear_rect': [_p, _p, _i64, _i64, _int, _p, _p, _i64, _p, _p, _p, _p],
    'exb_stencil_bilinear_curv': [_p, _p, _p, _i64, _i64, _p, _p, _i64, _p, _p, _p, _p],
    'exb_stencil_combine': [_p, _p, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i64, _int, _p, _p, _p],
    'exb_pool_trim': [C.c_uint64],
    'exb_gather_f64': [_p, _i64, _int, _p, _p, _int, _i64, _p, _p],
    'exb_gather_f32': [_p, _i64, _int, _p, _p, _int, _i64, _p, _p],
    'exb_split_mean_pert_f64': [_p, _p, _i64, _int, _p],
    'exb_split_mean_pert_f32': [_p, _p, _i64, _int, _p],
    'exb_inflate_f64': [_p, _i64, _int, _p, _i64, _i64, _p],
    'exb_inflate_f32': [_p, _i64, _int, _p, _i64, _i64, _p],
    'exb_recombine_f64': [_p, _p, _i64, _int, _p],
    'exb_recombine_f32': [_p, _p, _i64, _int, _p],
    'exb_row_spread_f64': [_p, _i64, _i64, _i64, _i64, _int, _p, _p],
    'exb_row_spread_f32': [_p, _i64, _i64, _i64, _i64, _int, _p, _p],
    'exb_relax_rtps_f64': [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _p],
    'exb_relax_rtps_f32': [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _p],
    'exb_relax_rtpp_f64': [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _p],
    'exb_relax_rtpp_f32': [_p, _p, _p, _i64, _i64, _i64, _i64, _int, _p],
    'exb_obs_solve_f64': [_p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_f32': [_p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_async_status': [],
    'exb_obs_plan_create': [_p, _p, _i64, _int, _p, _p],
    'exb_obs_plan_create_dist': [_p, _p, _i64, _int, _int, _int, _int, _p, _p],
    'exb_obs_plan_finish': [_p],
    'exb_obs_solve_dist_f64': [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _int, _int, _p, _p, _p],
    'exb_obs_solve_dist_f32': [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _int, _int, _p, _p, _p],
    'exb_obs_plan_destroy': [_p],
    'exb_obs_solve_planned_f64': [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_planned_f32': [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_qc_f64': [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_qc_f32': [_p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_planned_qc_f64': [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_planned_qc_f32': [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _p],
    'exb_obs_solve_dist_qc_f64': [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _int, _int, _p, _p, _p],
    'exb_obs_solve_dist_qc_f32': [_p, _p, _p, _p, _p, _p, _p, _p, _i64, _int, _int, _p, _p, _int, _int, _p, _p, _p],
    'exb_state_update_f64': [_p, _p, _i64, _i64, _i64, _int, _p, _p, _p, _p, _i64, _i64, _i64, _int, _p, _p],
    'exb_state_update_f32': [_p, _p, _i64, _i64, _i64, _int, _p, _p, _p, _p, _i64, _i64, _i64, _int, _p, _p],
    'exb_state_sweep_f64': [_p, _i64, _i64, _i64, _int, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i64, _int, _p, _p],
    'exb_state_sweep_f32': [_p, _i64, _i64, _i64, _int, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i64, _int, _p, _p],
    'exb_sweep_plan_create': [_p, _i64, _i64, _i64, _p, _p, _i64, _i64, _i64, _i64, _i64, _int, _p, _p],
    'exb_sweep_plan_destroy': [_p],
    'exb_state_sweep_planned_f64': [_p, _p, _i64, _i64, _i64, _int, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i64, _int, _p, _p],
    'exb_state_sweep_planned_f32': [_p, _p, _i64, _i64, _i64, _int, _p, _p, _p, _p, _i64, _i64, _i64, _i64, _i64, _int, _p, _p],
    'exb_localization_weights': [_p, _i64, _dbl, _dbl, _dbl, _int, _p, _p, _p],
    'exb_gaspari_cohn': [_p, _i64, _dbl, _p, _p],
    'exb_ensrf_host_f64': [_p, _i64, _i64, _i64, _int, _p, _p, _i64, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p,
                           _int, _dbl, _p, _p],
    'exb_measure_fp64_peak': [_p, _p],
    'exb_measure_dmma_peak': [_p, _p],
}

_lib = None


class ExbError(RuntimeError):
    """A call into libefa_xray_b200 returned a non-zero status."""


def load():
    """Load the shared library (once).  Raises ImportError with build instructions if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            'efa_xray_b200: CUDA library %s is not built.  Run `python -m efa_xray_b200._build` '
            '(needs nvcc; no GPU required to build).  There is no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export it
        fn.argtypes = argtypes
        fn.restype = _int
    lib.exb_state_sweep_row_granularity.argtypes = [_i64, _i64, _i64]
    lib.exb_state_sweep_row_granularity.restype = _int
    lib.exb_launch_count.argtypes = []
    lib.exb_launch_count.restype = C.c_int64
    lib.exb_last_error.argtypes = []
    lib.exb_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def call(name, *args):
    """Call a library function and raise ExbError on a non-zero status."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if rc != 0:
        raise ExbError('%s failed (%d): %s' % (name, rc, lib.exb_last_error().decode('utf-8', 'replace')))
    return rc


def launch_count():
    """Number of kernels this library has launched so far in this process."""
    return int(load().exb_launch_count())


def require_device():
    """Raise unless a usable sm_100 device is current."""
    import torch
    if not torch.cuda.is_available():
        raise ExbError('efa_xray_b200 needs a CUDA (sm_100a) device; torch.cuda.is_available() is False. '
                       'There is no CPU fallback.')
    call('exb_device_check')


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
