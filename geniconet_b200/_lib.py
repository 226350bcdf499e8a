"""ctypes binding of libgeniconet_b200.so (include/geniconet_b200.h).

There is no CPU implementation behind this module: if the shared library is missing it is
built with nvcc, and if that is impossible the import fails loudly.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('GIN_LIB') or os.path.join(_HERE, 'libgeniconet_b200.so')      # GIN_LIB: diagnostics builds (-DGIN_PROF)

PLAN_HEXCONV, PLAN_UPSAMPLE, PLAN_LOSS = 1, 2, 3
IMPL_AUTO, IMPL_SIMT, IMPL_TC = 0, 1, 2
ERR_UNSUPPORTED = -4
CORNER = {'zeros': 0, 'average': 1}


class GinError(RuntimeError):
    pass


def _load():
    # A missing library is built here; a library that is OLDER than its sources (digest stamp mismatch) is rebuilt when nvcc is
    # available and otherwise refused -- never loaded silently.  The build itself runs under a file lock, so the ranks of a
    # torchrun job do not race on the same output file.
    if not os.environ.get('GIN_LIB'):
        from . import build as _build
        if not os.path.exists(LIB_PATH) or not _build.is_current():
            _build.build()
    try:
        return ctypes.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise ImportError('geniconet_b200: cannot load %s (%s); there is no fallback path' % (LIB_PATH, e))


lib = _load()

_vp, _i, _i64, _u64, _f, _sz = (ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64, ctypes.c_float,
                                ctypes.c_size_t)
_SIGS = {
    'gin_version': (_i, []),
    'gin_forward_operand_is_fp16': (_i, []),
    'gin_last_error': (ctypes.c_char_p, []),
    'gin_launch_count': (_i64, []),
    'gin_index_map_len': (_i, [_i]),
    'gin_index_map': (_i, [_i, _vp]),
    'gin_ico_faces_len': (_i, [_i]),
    'gin_ico_faces': (_i, [_i, _vp]),
    'gin_ico_vertices': (_i, [_i, _vp]),
    'gin_plan_bytes': (_sz, [_i, _i, _i, _i]),
    'gin_plan_build': (_i, [_i, _i, _i, _i, _vp, _sz]),
    'gin_hexconv_packed_bytes': (_sz, [_i, _i]),
    'gin_hexconv_pack_weights': (_i, [_vp, _vp, _i, _i, _vp]),
    'gin_hexconv_pack_weights_bf16': (_i, [_vp, _i, _vp, _i, _vp, _i, _vp]),
    'gin_hexconv_pack_weights_bf16_multi': (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'gin_hexconv_fwd': (_i, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'gin_hexconv_narrow_stats_ws_bytes': (_sz, [_i]),
    'gin_hexconv_fwd_narrow_stats': (_i, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    'gin_hexconv_dgrad': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'gin_hexconv_wgrad_ws_bytes': (_sz, [_i, _i]),
    'gin_hexconv_wgrad': (_i, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'gin_cast_bf16_bytes': (_sz, [_i, _i, _i]),
    'gin_cast_bf16': (_i, [_vp, _vp, _i, _vp, _vp, _i, _i, _vp]),
    'gin_cast_bf16_colsum_ws_bytes': (_sz, [_i]),
    'gin_cast_bf16_colsum': (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    'gin_hexconv_fwd_bf16': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'gin_hexconv_stats_ws_bytes': (_sz, [_i]),
    'gin_hexconv_fwd_bf16_stats': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp]),
    'gin_hexconv_fwd_bf16_stats2': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    'gin_hexconv_affine_ring_bytes': (_sz, [_i, _i]),
    'gin_hexconv_fwd_affine': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i64, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'gin_bn_eval_consts': (_i, [_vp, _i, _i, _vp]),
    'gin_bn_stats_from_parts': (_i, [_vp, _i, _i64, _i64, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp]),
    'gin_bn_stats_from_parts2': (_i, [_vp, _i, _i64, _i64, _i, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp]),
    'gin_hexconv_dgrad_bf16': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'gin_hexconv_wgrad_bf16': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'gin_bn_ws_bytes': (_sz, [_i]),
    'gin_bn_stats': (_i, [_vp, _i64, _i64, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp]),
    'gin_bn_act_fwd': (_i, [_vp, _i64, _vp, _vp, _i64, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'gin_bn_act_bwd': (_i, [_vp, _i64, _vp, _vp, _i64, _i, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i, _i, _i, _i, _vp]),
    'gin_bn_pair_ws_bytes': (_sz, [_i]),
    'gin_bn_act_bwd_pair': (_i, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _i, _vp, _i, _i, _i, _i, _vp]),
    'gin_bn_eval_bwd_ws_bytes': (_sz, [_i]),
    'gin_bn_eval_bwd': (_i, [_vp, _i64, _vp, _vp, _i64, _i, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i, _i, _i, _i, _vp]),
    'gin_bn_eval_bwd_pair': (_i, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp, _vp, _i64, _i, _vp, _i, _i, _i, _i, _vp]),
    'gin_upsample_bf16':(_i, [_vp, _vp, _vp, _i, _vp, _vp, _i, _i, _vp]),
    'gin_upsample_fwd': (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp]),
    'gin_upsample_bwd': (_i, [_vp, _vp, _vp, _vp, _i, _i, _vp]),
    'gin_reparam_fwd': (_i, [_vp, _vp, _vp, _vp, _i64, _u64, _u64, _vp]),
    'gin_reparam_fwd_step': (_i, [_vp, _vp, _vp, _vp, _i64, _u64, _u64, _vp, _vp]),
    'gin_reparam_bwd': (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    'gin_kld_fwd': (_i, [_vp, _vp, _vp, _vp, _i64, _vp]),
    'gin_kld_bwd': (_i, [_vp, _vp, _vp, _f, _vp, _vp, _i64, _vp]),
    'gin_pole_vertices_fwd': (_i, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i, _i, _vp]),
    'gin_pole_vertices_bwd': (_i, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i, _i, _vp]),
    'gin_adam_chunk': (_i, []),
    'gin_adam_step': (_i, [_vp, _vp, _i, _i, _f, _vp, _f, _f, _f, _f, _vp, _vp]),
    'gin_head_ws_bytes': (_sz, []),
    'gin_head_fwd': (_i, [_vp, _vp, _vp, _vp, _i, _i64, _i, _i, _vp]),
    'gin_head_bwd': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i64, _i, _i, _vp]),
    'gin_point_mesh_ws_bytes': (_sz, [_i, _i]),
    'gin_point_mesh_distance': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    'gin_chamfer_ws_bytes': (_sz, [_i, _i, _i]),
    'gin_chamfer_fwd': (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'gin_chamfer_bwd': (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'gin_vertex_normals_fwd': (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    'gin_laplacian_fwd': (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    'gin_ring_ops_ws_bytes': (_sz, [_i, _i]),
    'gin_ring_ops_bwd': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    'gin_p2p_ws_bytes': (_sz, [_i, _i]),
    'gin_p2p_loss_fwd': (_i, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _f, _f, _f, _vp, _vp, _i, _vp]),
    'gin_p2p_loss_bwd': (_i, [_vp, _vp, _vp, _i64, _i64, _i64, _vp, _f, _f, _f, _vp, _vp, _vp, _i, _vp]),
}
EXPORTS = tuple(_SIGS)
for _name, (_res, _args) in _SIGS.items():
    _fn = getattr(lib, _name)          # AttributeError here == the .so does not match the header
    _fn.restype, _fn.argtypes = _res, _args


def check(rc, what=''):
    if rc != 0:
        raise GinError('%s failed (%d): %s' % (what or 'geniconet_b200 call', rc, lib.gin_last_error().decode()))


def forward_operand_dtype():
    """torch dtype of the forward-side 16-bit operand copies (fp16 by default, bf16 under GIN_FWD_FP16=0)."""
    import torch
    return torch.float16 if lib.gin_forward_operand_is_fp16() else torch.bfloat16


def launch_count():
    return int(lib.gin_launch_count())


# ---------------------------------------------------------------- host-side helpers
def index_map(level):
    """int32 [5, n+2, 2n+2] chart-padding index map (row a1)."""
    n = 2 ** level
    out = np.empty((5, n + 2, 2 * n + 2), dtype=np.int32)
    assert lib.gin_index_map_len(level) == out.size
    check(lib.gin_index_map(level, out.ctypes.data), 'gin_index_map')
    return out


def ico_faces(level):
    out = np.empty((lib.gin_ico_faces_len(level) // 3, 3), dtype=np.int32)
    check(lib.gin_ico_faces(level, out.ctypes.data), 'gin_ico_faces')
    return out


def ico_vertices(level):
    out = np.empty((10 * 4 ** level + 2, 3), dtype=np.float32)
    check(lib.gin_ico_vertices(level, out.ctypes.data), 'gin_ico_vertices')
    return out


def plan_blob(kind, level, stride=1, corner_mode='average'):
    """Host plan blob as an int32 numpy array."""
    cm = CORNER[corner_mode] if isinstance(corner_mode, str) else int(corner_mode)
    nbytes = lib.gin_plan_bytes(kind, level, stride, cm)
    if nbytes == 0:
        raise GinError('gin_plan_bytes: ' + lib.gin_last_error().decode())
    out = np.empty(nbytes // 4, dtype=np.int32)
    check(lib.gin_plan_build(kind, level, stride, cm, out.ctypes.data, nbytes), 'gin_plan_build')
    return out
