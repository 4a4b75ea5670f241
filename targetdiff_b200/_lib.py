"""ctypes binding of libtdiff.so (the C-ABI declared in include/tdiff.h).

There is no CPU or PyTorch fallback: if the shared library is missing, or a call fails, this module raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('TDIFF_LIB') or os.path.join(_HERE, 'libtdiff.so')      # TDIFF_LIB: developer switch (A/B of kernel builds)

TDIFF_OK, TDIFF_EINVAL, TDIFF_ECUDA, TDIFF_ESTATE, TDIFF_EWEIGHT = 0, -1, -2, -3, -4


class TdiffError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__('libtdiff error %d: %s' % (code, msg))
        self.code = code


class tdiff_config(ctypes.Structure):
    _fields_ = [('hidden_dim', ctypes.c_int32), ('n_heads', ctypes.c_int32), ('num_layers', ctypes.c_int32), ('knn', ctypes.c_int32),
                ('num_r_gaussian', ctypes.c_int32), ('num_classes', ctypes.c_int32), ('protein_feat_dim', ctypes.c_int32),
                ('num_timesteps', ctypes.c_int32), ('model_mean_type', ctypes.c_int32), ('num_blocks', ctypes.c_int32),
                ('ew_net_type', ctypes.c_int32), ('x2h_out_fc', ctypes.c_int32), ('time_emb', ctypes.c_int32), ('cutoff_mode', ctypes.c_int32),
                ('reserved', ctypes.c_int32 * 2)]


class tdiff_prop_config(ctypes.Structure):
    _fields_ = [('hidden_dim', ctypes.c_int32), ('num_layers', ctypes.c_int32), ('knn', ctypes.c_int32), ('num_r_gaussian', ctypes.c_int32),
                ('edge_dim', ctypes.c_int32), ('norm', ctypes.c_int32), ('protein_feat_dim', ctypes.c_int32), ('ligand_feat_dim', ctypes.c_int32),
                ('enc_ligand_dim', ctypes.c_int32), ('enc_node_dim', ctypes.c_int32), ('enc_graph_dim', ctypes.c_int32),
                ('output_dim', ctypes.c_int32), ('reserved', ctypes.c_int32 * 4)]


class tdiff_tensor(ctypes.Structure):
    _fields_ = [('name', ctypes.c_char_p), ('data', ctypes.c_void_p), ('numel', ctypes.c_int64)]


_vp, _i, _i64, _u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64
_pi32 = ctypes.POINTER(ctypes.c_int32)

# name -> (restype, argtypes); must list every symbol include/tdiff.h declares (tests/test_cabi_symbols.py checks)
SIGNATURES = {
    'tdiff_create': (_i, [ctypes.POINTER(tdiff_config), ctypes.POINTER(tdiff_tensor), _i, _i, ctypes.POINTER(_vp)]),
    'tdiff_destroy': (None, [_vp]),
    'tdiff_last_error': (ctypes.c_char_p, []),
    'tdiff_version': (ctypes.c_char_p, []),
    'tdiff_bind_batch': (_i, [_vp, _i, _pi32, _pi32, _vp, _vp, _i, _vp]),
    'tdiff_set_ligand': (_i, [_vp, _vp, _vp, _i, _vp]),
    'tdiff_get_ligand': (_i, [_vp, _vp, _vp, _i, _vp]),
    'tdiff_get_offset': (_i, [_vp, _vp, _vp]),
    'tdiff_set_time': (_i, [_vp, _vp, _vp]),
    'tdiff_forward': (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    'tdiff_num_edges': (_i64, [_vp, _vp]),
    'tdiff_get_edge_index': (_i, [_vp, _vp, _vp]),
    'tdiff_get_edge_weight': (_i, [_vp, _vp, _vp]),
    'tdiff_get_node_pos': (_i, [_vp, _vp, _vp]),
    'tdiff_sample': (_i, [_vp, _i, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _i, _vp]),
    'tdiff_sample_host': (_i, [_vp, _i, _pi32, _pi32, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _u64, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    'tdiff_knn_graph': (_i, [_vp, _i, _pi32, _i, _i, _vp, _vp, ctypes.POINTER(_i64), _vp]),
    'tdiff_attn_aggregate_h': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    'tdiff_attn_aggregate_x': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    'tdiff_scatter_mean3': (_i, [_vp, _pi32, _i, _vp, _vp]),
    'tdiff_check_stability': (_i, [_vp, _vp, _pi32, _i, _i, _vp, _vp, _vp, _vp]),
    'tdiff_prop_create': (_i, [ctypes.POINTER(tdiff_prop_config), ctypes.POINTER(tdiff_tensor), _i, _i, ctypes.POINTER(_vp)]),
    'tdiff_prop_destroy': (None, [_vp]),
    'tdiff_prop_forward': (_i, [_vp, _i, _pi32, _pi32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'tdiff_prop_profile': (_i, [_vp, _i]),
    'tdiff_prop_profile_read': (_i, [_vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    'tdiff_launch_count': (_i64, [_vp]),
    'tdiff_edge_mlp_mode': (_i, [_vp]),
    'tdiff_profile': (_i, [_vp, _i]),
    'tdiff_profile_read': (_i, [_vp, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(_i64), ctypes.POINTER(ctypes.c_double),
                                ctypes.POINTER(_i64), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(_i64), ctypes.POINTER(ctypes.c_double)]),
}

_lib = None


def load():
    """Load libtdiff.so (once).  Raises if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError('%s not found: build it with `python -m targetdiff_b200.build` (nvcc, sm_100a). '
                           'targetdiff_b200 has no CPU / PyTorch fallback.' % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().tdiff_last_error().decode('utf-8', 'replace')


def check(rc):
    if rc != TDIFF_OK:
        raise TdiffError(rc, last_error())


def i32_array(values):
    arr = (ctypes.c_int32 * len(values))(*[int(v) for v in values])
    return arr
