"""ctypes binding of libtriplane_b200.so (include/triplane_b200.h).

The library is prebuilt for sm_100a by ``build.py``; there is no fallback of any kind: if the
shared object is missing or fails to load, importing this module's ``lib()`` raises.
``bench_lib()`` binds the separate measurement library (include/triplane_b200_bench.h: gather / tcgen05.mma
microbenchmarks, the raw tcgen05 layer test); the renderer never loads it.
"""
import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int32, c_int64, c_size_t, c_void_p

from .build import LIB_PATH, BENCH_LIB_PATH

ABI_VERSION = 8
MLP_FP32, MLP_BF16, MLP_FFMA = 0, 1, 2
BWD_DETERMINISTIC = 0x100          # OR-ed into the flags of the two backward entry points (TPR_BWD_DETERMINISTIC)
LAYOUT_CHANNELS_LAST, LAYOUT_CHANNELS_FIRST = 0, 1


class TprOptions(ctypes.Structure):
    _fields_ = [('ray_start', c_double), ('ray_end', c_double), ('box_warp', c_double),
                ('depth_resolution', c_int32), ('depth_resolution_importance', c_int32),
                ('disparity_space_sampling', c_int32), ('white_back', c_int32),
                ('flags', c_int32), ('tile_width', c_int32), ('plane_sets', c_int32),
                ('output_layout', c_int32), ('depth_clamp_group', c_int32), ('reserved', c_int32),
                ('density_noise', c_double), ('density_noise_coarse', c_void_p), ('density_noise_fine', c_void_p)]


MAX_PEERS, PEER_HANDLE_BYTES = 15, 64


class TprPeerSinks(ctypes.Structure):
    _fields_ = [('n_peers', c_int32), ('reserved', c_int32), ('rgb', c_void_p * MAX_PEERS),
                ('depth', c_void_p * MAX_PEERS), ('weight_sum', c_void_p * MAX_PEERS)]


_P = c_void_p
_SIGNATURES = {
    'tpr_abi_version': (ctypes.c_int, []),
    'tpr_last_error': (c_char_p, []),
    'tpr_packed_planes_bytes': (c_size_t, [c_int64, c_int32, c_int32]),
    'tpr_pack_planes': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P]),
    'tpr_unpack_planes': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P]),
    'tpr_packed_decoder_bytes': (c_size_t, []),
    'tpr_pack_decoder': (ctypes.c_int, [_P, _P, _P, _P, c_float, c_float, c_float, c_float, _P, _P]),
    'tpr_ray_sample': (ctypes.c_int, [_P, _P, c_int64, c_int32, _P, _P, _P]),
    'tpr_run_model': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P, c_int64, c_double, _P, _P, c_int32, _P]),
    'tpr_decode': (ctypes.c_int, [_P, c_int64, c_int64, _P, _P, _P, c_int32, _P]),
    'tpr_render_scratch_bytes': (c_size_t, [c_int64, c_int64, ctypes.POINTER(TprOptions)]),
    'tpr_render': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P, _P, c_int64, _P, _P, _P, _P,
                                  ctypes.POINTER(TprOptions), _P, _P, _P, _P, _P, _P, c_int32, _P, c_size_t, _P]),
    'tpr_render_peers': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P, _P, c_int64, _P, _P, _P, _P,
                                        ctypes.POINTER(TprOptions), _P, _P, _P, _P, _P, c_size_t,
                                        ctypes.POINTER(TprPeerSinks), _P]),
    'tpr_peer_alloc': (ctypes.c_int, [c_size_t, ctypes.POINTER(c_void_p), ctypes.c_char_p]),
    'tpr_peer_open': (ctypes.c_int, [ctypes.c_char_p, ctypes.POINTER(c_void_p)]),
    'tpr_peer_close': (ctypes.c_int, [_P]),
    'tpr_peer_free': (ctypes.c_int, [_P]),
    'tpr_clamp_depth': (ctypes.c_int, [_P, c_int64, _P, _P]),
    'tpr_render_host_workspace_bytes': (c_size_t, [c_int64, c_int32, c_int32, c_int64]),
    'tpr_render_host': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P, _P, c_int64, _P, _P,
                                       ctypes.POINTER(TprOptions), _P, _P, _P, _P, _P, c_size_t, _P]),
    'tpr_render_host_depth': (ctypes.c_int, [_P, c_size_t, c_int64, c_int32, c_int32, c_int64, _P, _P, _P]),
    'tpr_ray_march': (ctypes.c_int, [_P, _P, _P, c_int64, c_int32, c_int32, c_int32, _P, _P, _P, _P, c_int32, _P]),
    'tpr_sample_importance': (ctypes.c_int, [_P, _P, _P, c_int64, c_int32, c_int32, _P, _P, _P]),
    'tpr_sample_pdf': (ctypes.c_int, [_P, c_int32, _P, _P, c_int64, c_int32, c_int32, _P, _P, _P]),
    'tpr_sample_stratified': (ctypes.c_int, [_P, c_int64, _P, _P, ctypes.POINTER(TprOptions), _P, _P]),
    'tpr_ray_limits_box': (ctypes.c_int, [_P, _P, c_int64, c_float, _P, _P, _P]),
    'tpr_render_backward_scratch_bytes': (c_size_t, [c_int64, c_int64, c_int32]),
    'tpr_render_backward': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P, _P, c_int64, _P, _P, _P,
                                           ctypes.POINTER(TprOptions), _P, _P, _P, _P, _P, _P, _P, _P, _P, c_size_t, _P]),
    'tpr_render_train': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P, _P, c_int64, _P, _P, _P, _P,
                                        ctypes.POINTER(TprOptions), _P, _P, _P, _P, _P, _P, _P, _P, ctypes.POINTER(c_int32), _P,
                                        c_size_t, _P]),
    'tpr_run_model_backward_scratch_bytes': (c_size_t, [c_int64, c_int64]),
    'tpr_run_model_backward': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, _P, c_int64, c_double, _P, _P, _P, c_int32,
                                              _P, _P, _P, c_size_t, _P]),
    'tpr_backward_deterministic_scratch_bytes': (c_size_t, [c_int64, c_int32, c_int32]),
    'tpr_unpack_decoder_grad': (ctypes.c_int, [_P, c_float, c_float, c_float, c_float, _P, _P, _P, _P, _P]),
    'tpr_march_backward': (ctypes.c_int, [_P, _P, c_int32, c_int32, _P, _P, _P, _P, _P, _P, c_int32, c_int64, _P, _P, _P]),
    'tpr_sample_planes': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, _P, c_int64, c_double, _P, _P]),
    'tpr_add_density_noise': (ctypes.c_int, [_P, _P, c_int64, c_double, _P]),
    'tpr_sort_samples': (ctypes.c_int, [_P, _P, _P, c_int64, c_int32, c_int32, _P, _P, _P, _P]),
    'tpr_sample_3dgrid': (ctypes.c_int, [_P, c_int64, c_int32, c_int32, c_int32, c_int32, _P, c_int64, c_int64, _P, _P]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)
_BENCH_SIGNATURES = {
    'tpr_gather_microbench': (c_int64, [_P, c_int64, c_int32, c_int32, _P, _P]),
    'tpr_mma_microbench': (ctypes.c_int, [c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    'tpr_gather_microbench_ex': (c_int64, [_P, c_int64, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    'tpr_gather_microbench_v2': (c_int64, [_P, c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    'tpr_scatter_microbench': (c_int64, [_P, c_int64, c_int32, c_int32, c_int32, c_int32, _P]),
    'tpr_debug_tc_decode': (ctypes.c_int, [_P, c_int64, _P, c_int32, _P, _P, _P]),
}
BENCH_EXPORTED_SYMBOLS = tuple(_BENCH_SIGNATURES)

_lib = None


def lib() -> ctypes.CDLL:
    """Load (once) and return the shared library; raise loudly if it is not there."""
    global _lib
    if _lib is None:
        path = os.environ.get('TPR_LIB') or LIB_PATH          # TPR_LIB: an A/B build made by build.py --alt (development aid)
        if not os.path.exists(path):
            raise RuntimeError(
                f'{path} is missing: the sm_100a CUDA library has not been built. Run '
                f'`python -c "import __graft_entry__ as g; g.build()"` (needs nvcc). There is no CPU or '
                f'PyTorch fallback for the tri-plane renderer.')
        handle = ctypes.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)           # AttributeError if a declared symbol is not exported
            fn.restype, fn.argtypes = res, args
        got = handle.tpr_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f'libtriplane_b200 ABI version {got}, binding expects {ABI_VERSION}: rebuild')
        _lib = handle
    return _lib


_bench = None


def bench_lib() -> ctypes.CDLL:
    """The measurement library (bench.py, profiles/, tests/test_gpu_tc_debug.py).  Not used by the renderer."""
    global _bench
    if _bench is None:
        if not os.path.exists(BENCH_LIB_PATH):
            raise RuntimeError(f'{BENCH_LIB_PATH} is missing: run `python -c "import __graft_entry__ as g; g.build()"`')
        handle = ctypes.CDLL(BENCH_LIB_PATH)
        for name, (res, args) in _BENCH_SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _bench = handle
    return _bench


def check(code: int, what: str) -> None:
    """Turn a non-zero C-ABI return into RuntimeError (the reference's plugins raise RuntimeError
    through TORCH_CHECK, torch_utils/ops/bias_act.cpp:39-55)."""
    if code != 0:
        msg = lib().tpr_last_error()
        raise RuntimeError(f'{what} failed (code {code}): {msg.decode() if msg else "?"}')
