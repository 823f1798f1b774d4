"""ctypes binding of the C-ABI in include/rua_b200.h (librua_b200.so, built by __graft_entry__.build()).

There is NO fallback: if the shared library is missing the import of any hot function raises, and
non-CUDA tensors are rejected by the callers in ``_native``.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_int32, c_int64, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'lib', 'librua_b200.so')

# enums (include/rua_b200.h)
CAT, LEFT, PACK, RIGHT = 0, 1, 2, 3
LEN_SAME, LEN_CONST, LEN_MINUS = 0, 1, 2
MAP_SHIFT, MAP_REV, MAP_ROLL = 0, 1, 2
PAD_FILL, PAD_ROW0, PAD_WRAP = 0, 1, 2
F32, F64, F16, BF16 = 0, 1, 2, 3
SUM, MEAN, PROD, MAX, MIN, LOGSUMEXP = 0, 1, 2, 3, 4, 5
SCAN_SUM, SCAN_LOGSUMEXP, SCAN_MAX, SCAN_MIN = 0, 1, 2, 3
CRF_FORWARD, CRF_BACKWARD, CRF_DECODE = 0, 1, 2


class Ragged(Structure):
    _fields_ = [('B', c_int64), ('off', c_void_p), ('poff', c_void_p), ('sorted', c_void_p),
                ('unsorted', c_void_p), ('Tp', c_int64)]


class Side(Structure):
    _fields_ = [('layout', c_int32), ('len_xform', c_int32), ('len_arg', c_int64), ('width', c_int64),
                ('rows', c_int64)]


# name -> (restype, argtypes); must list EVERY symbol include/rua_b200.h declares
SIGNATURES = {
    'rua_version': (c_int32, []),
    'rua_error_string': (c_char_p, [c_int32]),
    'rua_last_cuda_error': (c_int32, []),
    'rua_launch_count': (c_int64, []),
    'rua_selftest': (c_int32, []),
    'rua_scan_workspace_bytes': (c_size_t, [c_int64]),
    'rua_scan_lengths': (c_int32, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'rua_scan_lengths_ex': (c_int32, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p,
                                      c_int64, c_void_p, c_void_p, c_int64, c_void_p]),
    'rua_pinned_alloc': (c_int32, [c_size_t, POINTER(c_void_p), POINTER(c_void_p)]),
    'rua_pinned_free': (c_int32, [c_void_p]),
    'rua_sort_workspace_bytes': (c_size_t, [c_int64]),
    'rua_sort_lengths': (c_int32, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'rua_sort_keys': (c_int32, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    'rua_bucket_offsets': (c_int32, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    'rua_segment_reduce_gather': (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int32, c_int32,
                                            c_void_p, c_void_p, c_size_t, c_void_p]),
    'rua_invert_permutation': (c_int32, [c_void_p, c_int64, c_void_p, c_void_p]),
    'rua_batch_sizes': (c_int32, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    'rua_lengths_from_pack': (c_int32, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    'rua_meta_fused_max_batch': (c_int64, []),
    'rua_meta_fused': (c_int32, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                 c_void_p]),
    'rua_row_map': (c_int32, [c_void_p, c_void_p, c_int64, POINTER(Ragged), POINTER(Side), POINTER(Side),
                              c_int32, c_int64, c_int32, c_char_p, c_int32, c_void_p]),
    'rua_row_map_mask': (c_int32, [c_void_p, c_void_p, c_int64, POINTER(Ragged), POINTER(Side), POINTER(Side), c_char_p, c_int32,
                                   c_char_p, c_char_p, c_int32, c_void_p, c_void_p]),
    'rua_row_map_list': (c_int32, [c_void_p, c_int32, c_void_p, c_int64, POINTER(Ragged), POINTER(Side), c_char_p,
                                   c_int32, c_void_p]),
    'rua_gather_rows_multi': (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    'rua_gather_rows': (c_int32, [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    'rua_scatter_rows': (c_int32, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p]),
    'rua_token_rows': (c_int32, [POINTER(Ragged), POINTER(Side), c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    'rua_index_error_count': (c_int32, [POINTER(c_int64), c_int32]),
    'rua_mask': (c_int32, [c_void_p, c_int64, c_int64, c_char_p, c_char_p, c_int32, c_void_p, c_void_p]),
    'rua_emit_ptr': (c_int32, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                               c_int32, c_void_p]),
    'rua_segment_reduce_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int64, c_int32, c_int32]),
    'rua_segment_reduce': (c_int32, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int32, c_int32, c_void_p,
                                     c_void_p, c_size_t, c_void_p]),
    'rua_segment_reduce_strict': (c_int32, [c_void_p, c_void_p, c_int64, c_int64, c_int64, c_int32, c_int32, c_void_p,
                                            c_void_p]),
    'rua_segment_reduce_backward_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int64, c_int32, c_int32]),
    'rua_segment_reduce_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int64,
                                              c_int32, c_int32, c_void_p, c_void_p, c_size_t, c_void_p]),
    'rua_segment_scan_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int32, c_int32, c_int32]),
    'rua_segment_scan': (c_int32, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, POINTER(Ragged),
                                   POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_segment_scan_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32,
                                            c_int32, POINTER(Ragged), POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_segment_linrec_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int32, c_int32]),
    'rua_segment_linrec': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, POINTER(Ragged),
                                     POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_segment_linrec_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                              c_int64, c_int32, c_int32, POINTER(Ragged), POINTER(Side), c_void_p,
                                              c_size_t, c_void_p]),
    'rua_segment_conv_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int32, c_int32, c_int32]),
    'rua_segment_conv': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32,
                                   POINTER(Ragged), POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_segment_conv_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32,
                                            c_int32, c_int32, POINTER(Ragged), POINTER(Side), c_void_p, c_size_t,
                                            c_void_p]),
    'rua_crf_workspace_bytes': (c_size_t, [c_int64, c_int32, c_int32, c_int32]),
    'rua_crf_state_bytes': (c_size_t, [c_int64, c_int32, c_int32]),
    'rua_crf_forward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                  c_int32, POINTER(Ragged), POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_crf_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, POINTER(Ragged), POINTER(Side),
                                   c_void_p, c_size_t, c_void_p]),
    'rua_crf_decode': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, POINTER(Ragged),
                                 POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_ssm_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int64, c_int32, c_int32]),
    'rua_ssm_state_bytes': (c_size_t, [c_int64, c_int64, c_int64, c_int32, c_int32]),
    'rua_ssm_forward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int64, c_int32, c_int32, c_int32, POINTER(Ragged), POINTER(Side), c_void_p, c_size_t,
                                  c_void_p]),
    'rua_ssm_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32,
                                   POINTER(Ragged), POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_ssd_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int64, c_int64, c_int32, c_int32, c_int32, c_int32]),
    'rua_ssd_forward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int64, c_int32, c_int32, c_int32, c_int32, c_int32, POINTER(Ragged), POINTER(Side),
                                  c_void_p, c_size_t, c_void_p]),
    'rua_ssd_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32,
                                   c_int32, POINTER(Ragged), POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_gdn_workspace_bytes': (c_size_t, [c_int64, c_int64, c_int64, c_int64, c_int32, c_int32, c_int32, c_int32]),
    'rua_gdn_forward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int64, c_int32, c_int32, c_int32, c_double, c_int32, c_int32, POINTER(Ragged),
                                  POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_gdn_backward': (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_double,
                                   c_int32, c_int32, POINTER(Ragged), POINTER(Side), c_void_p, c_size_t, c_void_p]),
    'rua_peer_window_alloc': (c_int32, [c_size_t, POINTER(c_void_p), c_char_p]),
    'rua_peer_window_open': (c_int32, [c_char_p, POINTER(c_void_p)]),
    'rua_peer_window_close': (c_int32, [c_void_p]),
    'rua_peer_window_free': (c_int32, [c_void_p]),
    'rua_row_map_multi': (c_int32, [c_void_p, c_int64, POINTER(Ragged), POINTER(Side), c_int64, POINTER(c_void_p),
                                    POINTER(c_void_p), c_int32, c_void_p]),
    'rua_scatter_rows_multi': (c_int32, [c_void_p, c_void_p, c_int64, c_int64, POINTER(c_void_p), c_int32, c_void_p]),
}

MAX_DESTINATIONS = 16      # RUA_MAX_DESTINATIONS
PEER_HANDLE_BYTES = 64     # RUA_PEER_HANDLE_BYTES

_lib = None


def load() -> ctypes.CDLL:
    """Load librua_b200.so (once).  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'torchrua_b200: {LIB_PATH} is missing; build it with `python -c "import __graft_entry__ as g; '
                f'g.build()"` (nvcc, sm_100a).  There is no CPU / PyTorch fallback.')
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        lib = load()
        msg = lib.rua_error_string(status).decode()
        extra = f' (cudaError {lib.rua_last_cuda_error()})' if status == -4 else ''
        raise RuntimeError(f'torchrua_b200: {what} failed: {msg}{extra}')
