"""ctypes binding of libes_b200.so (C ABI declared in include/es_b200.h).

The library is the product: there is no Python/CPU fallback.  ``load()`` raises if the
shared object has not been built (``python -m es_pytorch_b200.build``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ES_B200_LIB: development override used by tools/ to time kernel variants built next to the product library
LIB_PATH = os.environ.get('ES_B200_LIB') or os.path.join(_HERE, 'libes_b200.so')

ES_RANK_CENTERED, ES_RANK_DOUBLE_POSITIVE, ES_RANK_SEMI_CENTERED, ES_RANK_MAX_NORMALIZED = 0, 1, 2, 3
ES_ROLLOUT_F32 = 0
ES_ROLLOUT_TC = 1
ES_ROLLOUT_TC3 = 2
ES_MT_N = 624

_vp, _i32, _i64, _u64, _f32, _f64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_float, C.c_double

# name -> (restype, argtypes); must list every symbol include/es_b200.h declares
SIGNATURES = {
    'es_ctx_create': (_i32, [_i32, C.POINTER(_vp)]),
    'es_ctx_destroy': (_i32, [_vp]),
    'es_last_error': (C.c_char_p, []),
    'es_abi_version': (_i32, []),
    'es_check_async': (_i32, [_vp]),
    'es_launch_count': (_i64, [_vp]),
    'es_noise_table_changed': (_i32, [_vp]),
    'es_sm_count': (_i32, [_vp]),
    'es_draw_indices': (_i32, [_vp, _vp, _vp, _i32, _i32, _u64, _i32, _vp, _vp, _vp]),
    'es_mt_skip': (_i32, [_vp, _vp, _vp, _i32, _i32, _vp]),
    'es_perturb': (_i32, [_vp, _vp, _vp, _i64, _vp, _i32, _i32, _f32, _vp, _vp, _vp]),
    'es_normalise_obs': (_i32, [_vp, _vp, _vp, _vp, _f64, _i32, _i32, _vp, _vp]),
    'es_rollout_openloop': (_i32, [_vp, _vp, _i64, _vp, _i32, _vp, _i32, _f32, C.POINTER(_i32), _i32, _vp, _vp, _i32,
                                   _f32, _vp, _vp, _i32, _vp, _vp, _i32, _vp]),
    'es_rollout_openloop_noisy': (_i32, [_vp, _vp, _i64, _vp, _i32, _vp, _i32, _f32, C.POINTER(_i32), _i32, _vp, _vp, _i32,
                                         _f32, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _vp]),
    'es_rollout_openloop_episodes': (_i32, [_vp, _vp, _i64, _vp, _i32, _vp, _i32, _f32, C.POINTER(_i32), _i32, _vp, _vp, _i32,
                                            _f32, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _i32, _vp]),
    'es_rollout_closedloop': (_i32, [_vp, _vp, _i64, _vp, _i32, _vp, _i32, _f32, C.POINTER(_i32), _i32, _vp, _vp, _f64, _vp, _vp, _i32,
                                     _vp, _vp, _i32, _f32, _vp, _f64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'es_draw_noisy': (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _u64, _i32, _i32, _f64, _vp, _vp, _vp, _vp]),
    'es_novelty': (_i32, [_vp, _vp, _i32, _vp, _i32, _i32, _vp, _i32, _vp]),
    'es_centered_rank': (_i32, [_vp, _vp, _vp, _i32, _i32, _f32, _f32, _i32, _i32, _vp, _vp, _vp]),
    'es_rank_transform': (_i32, [_vp, _vp, _vp, _i32, _i32, _i32, _f64, _f64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _vp, _vp]),
    'es_grad_reconstruct': (_i32, [_vp, _vp, _i64, _vp, _vp, _i32, _i32, _vp, _vp]),
    'es_adam_step': (_i32, [_vp, _vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _f32, _f32, _f32, _f32, _i32, _vp]),
    'es_sgd_step': (_i32, [_vp, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _f32, _i32, _vp]),
    'es_simple_step': (_i32, [_vp, _vp, _vp, _f32, _f32, _f32, _i32, _vp]),
    'es_obs_colsum': (_i32, [_vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    'es_obstat_accumulate': (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp]),
    'es_obstat_accumulate_coins': (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp, _i32, _f64, _vp]),
}

_lib = None


class EsLibraryError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load libes_b200.so and bind every entry point.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EsLibraryError(
            f'{LIB_PATH} not found: the CUDA library is the product path and there is no fallback. '
            f'Build it with `python -m es_pytorch_b200.build`.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = '') -> None:
    if rc != 0:
        msg = load().es_last_error()
        raise EsLibraryError(f'{what or "libes_b200"} failed (code {rc}): {msg.decode() if msg else "?"}')
