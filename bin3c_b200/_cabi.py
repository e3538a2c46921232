"""
ctypes binding of libbin3c_b200.so (include/bin3c_b200.h).

There is no CPU fallback: if the library has not been built, importing this module raises.
Build it with `python -m bin3c_b200.csrc.build` (or __graft_entry__.build()).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libbin3c_b200.so')

B3C_OK = 0
B3C_ERR_ARG = -1
B3C_ERR_CUDA = -2
B3C_ERR_CAPACITY = -3
B3C_ERR_NOCONV = -4
B3C_ERR_NAN = -5
B3C_ERR_TIE = -6
B3C_ERR_FORMAT = -7

B3C_EDGES_MAX_LINE_BYTES = 49     # the longest line b3c_edges_text writes


class B3CError(RuntimeError):
    """CUDA-side failure reported by the library."""


if not os.path.exists(LIB_PATH):
    raise ImportError('{} is missing: build the CUDA extension with '
                      '`python -m bin3c_b200.csrc.build` (there is no CPU fallback)'.format(LIB_PATH))

lib = C.CDLL(LIB_PATH)

_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64
_f64 = C.c_double
_pi64 = C.POINTER(C.c_int64)

# name: (restype, argtypes) -- must list every function declared in include/bin3c_b200.h
SIGNATURES = {
    'b3c_version': (C.c_int, []),
    'b3c_last_error': (C.c_char_p, []),
    'b3c_launch_count': (_i64, []),
    'b3c_accum_workspace_bytes': (_i64, [_i64, _i32, _i32]),
    'b3c_accum_begin': (C.c_int, [_p, _i64, _i64, _i32, _p, _i32, _p]),
    'b3c_accum_reset': (C.c_int, [_p, _p]),
    'b3c_accum_add_pairs': (C.c_int, [_p, _p, _i64, _p]),
    'b3c_accum_add_pairs_packed': (C.c_int, [_p, _p, _i64, _i32, _p]),
    'b3c_accum_add_pairs_same': (C.c_int, [_p, _p, _i64, _i32, _p]),
    'b3c_accum_reduce': (C.c_int, [_p, _pi64, _p]),
    'b3c_accum_emit_csr': (C.c_int, [_p, C.c_int, _p, _p, _p, _p]),
    'b3c_accum_offsets': (C.c_int, [_p, _pi64]),
    'b3c_accum_row_hist': (C.c_int, [_p, _p, _p]),
    'b3c_accum_route': (C.c_int, [_p, _p, _i32, _p, _i64, _p, _pi64, _p]),
    'b3c_accum_reduce_block': (C.c_int, [_p, _p, _i64, _i32, _i32, _pi64, _p]),
    'b3c_accum_emit_block': (C.c_int, [_p, _i32, _i32, _p, _p, _p, _p]),
    'b3c_max_offdiag_u32': (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p]),
    'b3c_max_offdiag_f64': (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p]),
    'b3c_acceptance_mask': (C.c_int, [_i32, _p, _p, _i64, _i64, _p, _p]),
    'b3c_site_norm': (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p]),
    'b3c_site_norm_f64': (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p]),
    'b3c_kr_workspace_bytes': (_i64, [_i32, _i64]),
    'b3c_kr_run': (C.c_int, [_i32, _i64, _p, _p, _p, _f64, _f64, _f64, _i32, _i32, _p, _p, _i64, _pi64, _p]),
    'b3c_kr_run_counts': (C.c_int, [_i32, _i64, _p, _p, _p, _p, _f64, _f64, _f64, _i32, _p, _p, _i64, _pi64, _p]),
    'b3c_krp_workspace_bytes': (_i64, [_i32, _i64]),
    'b3c_krp_setup': (C.c_int, [_i32, _i32, _i32, _i64, _p, _p, _p, _f64, _f64, _f64, _i32, _p, _i64, _pi64, _p]),
    'b3c_krp_phase': (C.c_int, [_p, _i32, _p]),
    'b3c_krp_scalar': (C.c_int, [_p, _i32, _p]),
    'b3c_krp_state': (C.c_int, [_p, _pi64, _p]),
    'b3c_kr_scale': (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p]),
    'b3c_asymmetry_count': (C.c_int, [_i32, _p, _p, _p, _f64, _p, _pi64, _p]),
    'b3c_spmv': (C.c_int, [_i32, _i64, _p, _p, _p, _p, _p, _p, _i64, _i32, _p]),
    'b3c_set_option': (C.c_int, [_i32, _i64]),
    'b3c_accum_plan': (C.c_int, [_i64, _i32, _i32, _pi64]),
    'b3c_peer_alloc': (C.c_int, [_i64, C.POINTER(C.c_void_p), C.c_char_p]),
    'b3c_peer_open': (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    'b3c_peer_close': (C.c_int, [_p]),
    'b3c_peer_free': (C.c_int, [_p]),
    'b3c_kr_exchange_bytes': (_i64, [_i32]),
    'b3c_kr_run_peer': (C.c_int, [_i32, _i32, _i32, _i64, _p, _p, _p, _f64, _f64, _f64, _i32, _i32, _i32,
                                  C.POINTER(C.c_void_p), _p, _p, _i64, _pi64, _p]),
    'b3c_kr_run_peer_counts': (C.c_int, [_i32, _i32, _i32, _i64, _p, _p, _p, _p, _f64, _f64, _f64, _i32, _i32, _i32,
                                         C.POINTER(C.c_void_p), _p, _p, _i64, _pi64, _p]),
    'b3c_xa_bytes': (_i64, [_i32, _i64]),
    'b3c_xa_offsets': (C.c_int, [_i32, _i64, _pi64]),
    'b3c_peer_barrier': (C.c_int, [C.POINTER(C.c_void_p), _i32, _i32, _i32, _i64, C.c_uint64, _p]),
    'b3c_peer_put': (C.c_int, [C.POINTER(C.c_void_p), _i32, _i64, _p, _i64, _p]),
    'b3c_peer_allreduce_f64': (C.c_int, [C.POINTER(C.c_void_p), _i32, _i32, _i32, _i64, C.c_uint64, _i32, _p, _i32, _p]),
    'b3c_shard_publish': (C.c_int, [_p, C.POINTER(C.c_void_p), _i32, _i32, _p]),
    'b3c_shard_scatter': (C.c_int, [_p, C.POINTER(C.c_void_p), _i32, _i32, _p, _p]),
    'b3c_shard_reduce_block': (C.c_int, [_p, C.POINTER(C.c_void_p), _i32, _i32, _p, _pi64, _p]),
    'b3c_compress_workspace_bytes': (_i64, [_i32]),
    'b3c_compress_count': (C.c_int, [_i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _i64, _p, _pi64, _p]),
    'b3c_compress_fill': (C.c_int, [_i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, C.c_int, _p, _p, _p, _p, _p, _p, _p,
                                    _p]),
    'b3c_edges_count': (C.c_int, [_i32, _i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _pi64, _p]),
    'b3c_edges_fill': (C.c_int, [_i32, _i32, _i32, _p, _p, _p, _p, _p, C.c_int, _p, _p, _p, _p, _p]),
    'b3c_extent_norm': (C.c_int, [_i32, _i32, _p, _p, _p, _p, _i32, _p, _p]),
    'b3c_synth_pairs': (C.c_int, [_p, _p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _f64, _f64, _f64, _f64, C.c_uint64,
                                  C.c_uint64, _i64, _p, _p]),
    'b3c_bamdec_workspace_bytes': (_i64, [_i32, _i32]),
    'b3c_bamdec_begin': (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _i32, _i64, _p]),
    'b3c_bamdec_slab': (C.c_int, [_p, _p, _p, _i32, _i64, _i64, _p, _i64, _p, _i64, _i32, _p, _i64, _pi64, _p]),
    'b3c_bamdec_stats': (C.c_int, [_p, _pi64, _i32, _p]),
    'b3c_sites_workspace_bytes': (_i64, [_i64, _i32]),
    'b3c_sites_begin': (C.c_int, [_p, _i64, _i64, _p, _p, _p, _i32, _i32, _p]),
    'b3c_sites_slab': (C.c_int, [_p, _p, _i64, _p, _i64, _p, _i64, _pi64, _p]),
    'b3c_sites_finish': (C.c_int, [_p, _p, _p, _i64, _pi64, _p]),
    'b3c_edges_text_workspace_bytes': (_i64, [_i64]),
    'b3c_edges_text': (C.c_int, [_p, _i64, _p, _p, _p, _i64, _i32, _i32, _p, _i64, _pi64, _p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)          # AttributeError here == the .so is stale: rebuild
    _fn.restype = _res
    _fn.argtypes = _args


# test / debugging hook: a shorter cross-GPU wait than the default 60 s (include/bin3c_b200.h: B3C_OPT_PEER_TIMEOUT_MS)
if os.environ.get('B3C_PEER_TIMEOUT_MS'):
    lib.b3c_set_option(4, int(os.environ['B3C_PEER_TIMEOUT_MS']))


def last_error():
    return lib.b3c_last_error().decode('utf-8', 'replace')


def check(rc):
    """Map a b3c_status to the exception type the reference raises for the same condition."""
    if rc == B3C_OK:
        return
    msg = last_error()
    if rc == B3C_ERR_ARG:
        raise AssertionError(msg)                   # the reference asserts on bad arguments
    if rc == B3C_ERR_TIE:
        raise ValueError(msg)                       # np.amin of an empty selection (Q13)
    if rc == B3C_ERR_FORMAT:
        raise ValueError(msg)                       # malformed BAM file: what the host reader raises for it
    if rc in (B3C_ERR_NOCONV, B3C_ERR_NAN):
        raise RuntimeError(msg)                     # sparse_utils.py:193,214
    raise B3CError('b3c status {}: {}'.format(rc, msg))


def launch_count():
    return int(lib.b3c_launch_count())
