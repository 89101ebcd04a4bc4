"""ctypes binding of libobe_b200.so (include/obe_b200.h).

The shared library is built in-tree by ``optbayesexpt_b200.build`` (nvcc, sm_100a).  There is no
CPU implementation behind these symbols: a missing library or a machine without a CUDA device
raises, it never falls back.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('OBE_B200_LIB', os.path.join(HERE, 'libobe_b200.so'))   # override: A/B builds

TILE = 2048
STATS_LEN = 64
PLAN_LEN = 512
PLAN_GSTATS, PLAN_COUNTS, PLAN_OVERFLOW = 352, 416, 9
MAX_PARAMS = 8
MAX_DRAWS = 128
MAX_CHANNELS = 4
MAX_SETTINGS = 4
MAX_CONSTANTS = 8

ST_TOTAL, ST_INVS, ST_SUMSQ, ST_NEFF = 0, 1, 2, 3
ST_M1, ST_M2, ST_PIVOT, ST_NOISE, ST_SUMT, ST_NZERO, ST_UNIFORM, ST_FIRED = 4, 12, 48, 56, 60, 61, 62, 63
MULTI_MAX = 128


class ObeError(RuntimeError):
    pass


class Cloud(C.Structure):
    _fields_ = [('particles_dev', C.c_void_p), ('weights_dev', C.c_void_p),
                ('tile_sums_dev', C.c_void_p), ('tile_prefix_dev', C.c_void_p),
                ('stats_dev', C.c_void_p), ('scratch_dev', C.c_void_p),
                ('n', C.c_int64), ('ld', C.c_int64), ('d', C.c_int32), ('reserved', C.c_int32),
                ('n_dev', C.c_void_p)]


class Batch(C.Structure):
    _fields_ = [('particles_dev', C.c_void_p * 2), ('weights_dev', C.c_void_p * 2), ('cur_dev', C.c_void_p),
                ('tile_sums_dev', C.c_void_p), ('tile_prefix_dev', C.c_void_p), ('stats_dev', C.c_void_p),
                ('pivot_dev', C.c_void_p), ('record_dev', C.c_void_p), ('last_idx_dev', C.c_void_p),
                ('best_val_dev', C.c_void_p), ('flag_dev', C.c_void_p), ('list_dev', C.c_void_p),
                ('n_list_dev', C.c_void_p), ('epoch_dev', C.c_void_p),
                ('n_inst', C.c_int64), ('n', C.c_int64), ('np', C.c_int64), ('ld', C.c_int64),
                ('d', C.c_int32), ('tiles', C.c_int32)]


class Cycle(C.Structure):
    """obe_cycle_t (include/obe_b200.h): one whole cycle in one C call."""
    _fields_ = [('model', C.c_void_p), ('cloud', C.POINTER(Cloud)), ('alt', C.POINTER(Cloud)),
                ('constants', C.POINTER(C.c_double)),
                ('setting', C.c_double * MAX_SETTINGS), ('y_meas', C.c_double * MAX_CHANNELS),
                ('sigma', C.c_double * MAX_CHANNELS), ('pivot', C.c_double * MAX_PARAMS),
                ('noise_index', C.c_int32 * MAX_CHANNELS),
                ('has_sigma', C.c_int32), ('has_noise_index', C.c_int32), ('n_lik_channels', C.c_int32),
                ('use_choke', C.c_int32), ('choke', C.c_double),
                ('resample', C.c_int32), ('scale', C.c_int32), ('u0', C.c_double), ('a_param', C.c_double),
                ('seed', C.c_uint64), ('epoch', C.c_uint32), ('mask_le', C.c_uint32), ('mask_lt', C.c_uint32),
                ('n_noise', C.c_int32),
                ('plan_dev', C.c_void_p), ('peer_bufs', C.POINTER(C.c_void_p)), ('rank', C.c_int32), ('world', C.c_int32),
                ('epoch_stats', C.c_uint64), ('epoch_draws', C.c_uint64), ('n_total', C.c_int64),
                ('select', C.c_int32), ('k', C.c_int32), ('u', C.c_double * 128), ('draws_dev', C.c_void_p),
                ('settings_dev', C.c_void_p), ('lds', C.c_int64), ('n_settings', C.c_int64),
                ('var_noise', C.c_double * MAX_CHANNELS), ('noise_from_stats', C.c_int32),
                ('method', C.c_int32), ('log_form', C.c_int32), ('pad0', C.c_int32),
                ('cost_dev', C.c_void_p), ('kld_noise_dev', C.c_void_p), ('utility_dev', C.c_void_p),
                ('best_dev', C.c_void_p), ('select_scratch_dev', C.c_void_p),
                ('stream', C.c_void_p), ('side_stream', C.c_void_p),
                ('resample_threshold', C.c_double), ('stats_host', C.c_void_p), ('stats_src_dev', C.c_void_p),
                ('best_host', C.c_void_p), ('phase', C.c_int32), ('pad1', C.c_int32),
                ('seq', C.c_uint64), ('seq_host', C.c_void_p)]


_PD = C.POINTER(C.c_double)
_PI32 = C.POINTER(C.c_int32)
_PCLOUD = C.POINTER(Cloud)
_PBATCH = C.POINTER(Batch)
_VP = C.c_void_p

# name -> (restype, argtypes); every symbol include/obe_b200.h declares
SIGNATURES = {
    'obe_abi_version': (C.c_int, []),
    'obe_last_error': (C.c_char_p, []),
    'obe_device_count': (C.c_int, []),
    'obe_set_option': (C.c_int, [C.c_char_p, C.c_int64]),
    'obe_num_tiles': (C.c_int64, [C.c_int64]),
    'obe_scratch_bytes': (C.c_size_t, [C.c_int64]),
    'obe_select_scratch_bytes': (C.c_size_t, [C.c_int64]),
    'obe_model_builtin': (C.c_int, [C.c_char_p, C.c_int, C.POINTER(_VP)]),
    'obe_model_compile': (C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                    C.POINTER(_VP), C.c_char_p, C.c_size_t]),
    'obe_model_compile_likelihood': (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(_VP),
                                               C.c_char_p, C.c_size_t]),
    'obe_model_compile_likelihood_design': (C.c_int, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int,
                                                      C.c_int, C.c_int, C.c_char_p, C.c_char_p, C.c_char_p,
                                                      C.c_char_p, C.POINTER(_VP), C.c_char_p, C.c_size_t]),
    'obe_model_info': (C.c_int, [_VP] + [C.POINTER(C.c_int)] * 5),
    'obe_model_free': (None, [_VP]),
    'obe_set_uniform': (C.c_int, [_PCLOUD, _VP]),
    'obe_update': (C.c_int, [_VP, _PCLOUD, _PD, _PD, _PD, _PD, _PI32, C.c_int, C.c_int, C.c_double, _PD, _VP]),
    'obe_update_from_y': (C.c_int, [_PCLOUD, _VP, C.c_int64, C.c_int, _PD, _PD, _PI32, C.c_int, C.c_int,
                                    C.c_double, _PD, _VP]),
    'obe_update_from_y_model': (C.c_int, [_VP, _PCLOUD, _VP, C.c_int64, C.c_int, _PD, _PD, _PI32, C.c_int, C.c_int,
                                          C.c_double, _PD, _VP]),
    'obe_update_from_likelihood': (C.c_int, [_PCLOUD, _VP, _PD, _VP]),
    'obe_refresh': (C.c_int, [_PCLOUD, C.c_uint32, C.c_uint32, _PI32, C.c_int, _PD, C.c_int, _VP]),
    'obe_fetch_stats': (C.c_int, [_PCLOUD, _PD, _VP]),
    'obe_materialize_weights': (C.c_int, [_PCLOUD, _VP]),
    'obe_normalized_weights': (C.c_int, [_PCLOUD, _VP, _VP]),
    'obe_summary_passes': (C.c_int, []),
    'obe_quantile_scratch_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'obe_histogram_scratch_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'obe_histogram2d_scratch_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'obe_quantile': (C.c_int, [_PCLOUD, _PI32, C.c_int, _PD, C.c_int, _VP, _PD, _VP]),
    'obe_summary_range': (C.c_int, [_PCLOUD, _PI32, C.c_int, _VP, _PD, _PD, _VP]),
    'obe_histogram': (C.c_int, [_PCLOUD, _PI32, C.c_int, _PD, C.c_int, _VP, C.POINTER(C.c_uint64),
                                C.POINTER(C.c_uint64), _VP]),
    'obe_histogram2d': (C.c_int, [_PCLOUD, C.c_int, C.c_int, _PD, C.c_int, _PD, C.c_int, _VP,
                                  C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), _VP]),
    'obe_cdf': (C.c_int, [_PCLOUD, _VP, _VP]),
    'obe_search': (C.c_int, [_PCLOUD, _VP, _VP, C.c_int64, _VP, _VP]),
    'obe_draw': (C.c_int, [_PCLOUD, _PD, C.c_int, _VP, _VP, _VP]),
    'obe_gather_jitter': (C.c_int, [_PCLOUD, _PCLOUD, _VP, _PD, _PD, _VP, C.c_uint64, C.c_uint32,
                                    C.c_double, C.c_int, _VP]),
    'obe_resample_systematic': (C.c_int, [_PCLOUD, _PCLOUD, C.c_double, _PD, _PD, C.c_uint64, C.c_uint32,
                                          C.c_double, C.c_int, _VP, _VP, _VP]),
    'obe_resample_systematic_sharded': (C.c_int, [_PCLOUD, _PCLOUD, C.c_double, C.c_int64, C.c_int64, C.c_int64,
                                                  C.c_double, C.c_double, C.c_int, _PD, _PD, C.c_uint64, C.c_uint32,
                                                  C.c_double, C.c_int, _VP, _VP, _VP]),
    'obe_shard_plan': (C.c_int, [_VP, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int64, C.c_double, C.c_int,
                                 _PCLOUD, _PCLOUD, _VP, _VP]),
    'obe_resample_systematic_planned': (C.c_int, [_PCLOUD, _PCLOUD, _VP, C.c_int64, C.c_uint64, C.c_uint32,
                                                  C.c_double, C.c_int, _VP]),
    'obe_draw_planned': (C.c_int, [_PCLOUD, _PD, C.c_int, _VP, _VP, C.c_int, _VP]),
    'obe_peer_bytes': (C.c_size_t, []),
    'obe_peer_alloc': (C.c_int, [C.POINTER(_VP), C.c_char_p]),
    'obe_peer_open': (C.c_int, [C.c_char_p, C.POINTER(_VP)]),
    'obe_peer_close': (C.c_int, [_VP]),
    'obe_peer_free': (C.c_int, [_VP]),
    'obe_shard_plan_peer': (C.c_int, [C.POINTER(_VP), C.c_int, C.c_int, C.c_uint64, C.c_int, C.c_double, C.c_int64,
                                      C.c_double, C.c_int, _PCLOUD, _PCLOUD, _VP, _VP]),
    'obe_cycle': (C.c_int, [C.POINTER(Cycle)]),
    'obe_stream_sync': (C.c_int, [_VP]),
    'obe_resample_defer': (C.c_int, [C.c_int]),
    'obe_resample_pick': (C.c_int, [_PD, C.c_int, _VP, C.POINTER(_VP), C.c_int, C.c_int, C.c_uint64, _VP]),
    'obe_resample_emit': (C.c_int, [_VP]),
    'obe_stream_fork': (C.c_int, [_VP, _VP]),
    'obe_stream_join': (C.c_int, [_VP, _VP]),
    'obe_draw_planned_peer': (C.c_int, [_PCLOUD, _PD, C.c_int, C.POINTER(_VP), C.c_int, C.c_int, C.c_uint64, _VP, C.c_int,
                                        _VP, _VP]),
    'obe_set_uniform_total': (C.c_int, [_PCLOUD, C.c_int64, _VP]),
    'obe_comb_count': (C.c_int64, [C.c_double, C.c_double, C.c_int64]),
    'obe_draw_strided': (C.c_int, [_PCLOUD, _PD, C.c_int, _VP, C.c_int, _VP, _VP]),
    'obe_utility': (C.c_int, [_VP, _VP, C.c_int, _VP, C.c_int64, C.c_int64, _PD, _PD, _VP, _VP, C.c_int,
                              C.c_int, _VP, _VP, _VP, _VP, _VP]),
    'obe_pick': (C.c_int, [_VP, C.c_int64, C.c_double, C.c_double, _VP, _VP, _VP]),
    'obe_batch_simulate': (C.c_int, [_VP, _PBATCH, _VP, C.c_int64, _VP, C.c_int64, _PD, _PD, _VP, C.c_uint64,
                                     C.c_uint32, C.c_int, _VP]),
    'obe_update_multi': (C.c_int, [_VP, _PCLOUD, _VP, _VP, C.c_int, _PD, _PI32, C.c_int, _PD, C.c_int, C.c_double,
                                   C.c_double, C.c_int64, _VP, _VP, _VP]),
    'obe_sweep_utility': (C.c_int, [_VP, C.c_int64, _VP, C.c_int64, C.c_double, _VP, _VP, _VP, _VP, _VP]),
    'obe_batch_init': (C.c_int, [_PBATCH, _PI32, C.c_int, _VP]),
    'obe_batch_update': (C.c_int, [_VP, _PBATCH, _VP, C.c_int64, C.c_int, _PD, _PI32, C.c_int, C.c_int, C.c_double,
                                   C.c_double, C.c_int, _VP]),
    'obe_batch_resample': (C.c_int, [_PBATCH, C.c_double, C.c_int, C.c_uint64, C.c_uint64, C.c_uint32, C.c_int,
                                     C.c_uint32, C.c_uint32, _PI32, C.c_int, _VP]),
    'obe_batch_refresh': (C.c_int, [_PBATCH, C.c_uint32, C.c_uint32, _PI32, C.c_int, _VP]),
    'obe_batch_select': (C.c_int, [_VP, _PBATCH, _VP, C.c_int64, C.c_int64, _PD, C.c_int, _PD, C.c_double,
                                   C.c_uint64, C.c_uint32, C.c_int, C.c_int, _VP, _VP]),
    'obe_eval_parameters': (C.c_int, [_VP, _PCLOUD, _PD, _PD, _VP, C.c_int64, _VP]),
    'obe_eval_settings': (C.c_int, [_VP, _VP, C.c_int64, C.c_int64, _PD, _PD, _VP, C.c_int64, _VP]),
}

_lib = None


def load():
    """Load libobe_b200.so (building it is the caller's job: ``python -m optbayesexpt_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ObeError(f'{LIB_PATH} is missing: run `python -m optbayesexpt_b200.build` '
                       '(there is no CPU fallback)')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.obe_abi_version() != 1:
        raise ObeError('libobe_b200.so ABI version mismatch: rebuild')
    # tuning knobs from the environment: OBE_OPT_PLAN_CLUSTER_MIN_TILES=..., OBE_OPT_UTILITY_LANE_FILL=...
    for key, val in os.environ.items():
        if key.startswith('OBE_OPT_'):
            if lib.obe_set_option(key[8:].lower().encode(), int(val)) != 0:
                raise ObeError(lib.obe_last_error().decode(errors='replace'))
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise ObeError(load().obe_last_error().decode(errors='replace'))


def darr(values, n=None):
    """Host double array for a by-value kernel argument (or None), zero-padded to n entries."""
    if values is None:
        return None
    a = np.ascontiguousarray(values, dtype=np.float64).reshape(-1)
    m = a.shape[0]
    out = (C.c_double * max(m, n or 0, 1))()
    if m:
        C.memmove(out, a.ctypes.data, 8 * m)
    return out


def dptr(array):
    """Pointer to a contiguous float64 numpy array (no copy; the array must outlive the call)."""
    return array.ctypes.data_as(_PD)


def raw_stream(torch, device_index=None):
    """The current CUDA stream as a void*; uses torch's raw accessor when it exists (it is several times
    cheaper than going through torch.cuda.current_stream(), and this runs four times per cycle).  Engines pass the
    index of the device they live on (it must be the current one, models.resolve_device), which saves the
    current_device() lookup -- a third of the host time of a small-cloud cycle went there."""
    get = getattr(torch._C, '_cuda_getCurrentRawStream', None)
    if get is not None:
        return C.c_void_p(get(torch.cuda.current_device() if device_index is None else device_index))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class ArgArray:
    """A reusable host double array for a by-value kernel argument: fill() overwrites the leading entries in place
    (no allocation, no numpy round trip per call)."""

    def __init__(self, n):
        self.n = n
        self.buf = (C.c_double * n)()

    def fill(self, values):
        buf = self.buf
        try:
            m = len(values)
        except TypeError:
            buf[0] = values
            return buf
        for i in range(m if m < self.n else self.n):
            buf[i] = values[i]
        return buf


def iarr(values):
    if values is None:
        return None
    vals = [int(v) for v in values]
    return (C.c_int32 * max(len(vals), 1))(*vals)


def require_device():
    lib = load()
    if lib.obe_device_count() <= 0:
        raise ObeError('no CUDA device visible: optbayesexpt_b200 has no CPU fallback')
    return lib
