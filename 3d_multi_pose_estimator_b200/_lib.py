"""ctypes binding of libb200pose.so (include/b200pose.h). The product path has no CPU fallback: if the
library is missing, or a call fails, a Python exception is raised."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libb200pose.so')

EXPORTS = ['b200pose_last_error', 'b200pose_version', 'b200pose_device_cc', 'b200pose_build_graph',
           'b200pose_node_features', 'b200pose_linear', 'b200pose_split_planes', 'b200pose_gat_aggregate', 'b200pose_gat_aggregate_res',
           'b200pose_cluster', 'b200pose_cluster_pairs', 'b200pose_build_graph_pairs', 'b200pose_encode_persons', 'b200pose_triangulate', 'b200pose_gather_persons',
           'b200pose_set_debug', 'b200pose_pack_record', 'b200pose_linear_n', 'b200pose_linear_fused2', 'b200pose_encode_persons_n', 'b200pose_pack_json', 'b200pose_packed_sizes', 'b200pose_packed_copy', 'b200pose_packed_free',
           'b200pose_gat_aggregate_bwd', 'b200pose_grad_planes', 'b200pose_transpose_planes', 'b200pose_colsum',
           'b200pose_mse_sigmoid', 'b200pose_sigmoid_bwd', 'b200pose_adam_step_dev',
           'b200pose_gat_prepare_layer', 'b200pose_gat_attn_bias_grad', 'b200pose_residual_bwd_add', 'b200pose_mlp_adam_planes']


class Cameras(C.Structure):
    """b200pose_cameras (include/b200pose.h)."""
    _fields_ = [('n_cameras', C.c_int32), ('v_sm', C.c_int32), ('v_pe', C.c_int32),
                ('image_width', C.c_float), ('image_height', C.c_float),
                ('sm_slot', C.c_void_p), ('pe_slot', C.c_void_p), ('kinv32', C.c_void_p),
                ('t_cam2root32', C.c_void_p), ('k64', C.c_void_p), ('dist64', C.c_void_p), ('p64', C.c_void_p),
                ('t_cam2root32_sm', C.c_void_p)]


class MlpLayer(C.Structure):
    """b200pose_mlp_layer (include/b200pose.h)."""
    _fields_ = [('offset', C.c_int64), ('n', C.c_int32), ('k', C.c_int32), ('ld', C.c_int32),
                ('w_hi', C.c_void_p), ('w_lo', C.c_void_p), ('ld_w', C.c_int32),
                ('wt_hi', C.c_void_p), ('wt_lo', C.c_void_p), ('ld_wt', C.c_int32)]


class B200PoseError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError('libb200pose.so not found at %s - build it with '
                              '`python 3d_multi_pose_estimator_b200/build.py` (there is no CPU fallback)' % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.b200pose_last_error.restype = C.c_char_p
        i32, f32, f64, vp = C.c_int32, C.c_float, C.c_double, C.c_void_p
        camp = C.POINTER(Cameras)
        L.b200pose_build_graph.argtypes = [i32, vp, vp, vp, camp, vp, vp, vp, vp, vp, vp, vp]
        L.b200pose_node_features.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, vp, camp, vp, i32, vp, vp, i32, vp]
        L.b200pose_linear.argtypes = [vp, vp, i32, vp, vp, i32, vp, i32, i32, i32, f32, f32, vp, i32, vp, vp, i32, i32, vp]
        L.b200pose_linear_n.argtypes = [vp, vp, i32, vp, vp, i32, vp, i32, vp, i32, i32, f32, f32, vp, i32, vp, vp, i32, i32, vp]
        L.b200pose_linear_fused2.argtypes = [vp, vp, i32, vp, vp, i32, vp, i32, i32, i32, f32, vp, i32, vp, i32, vp, i32, vp]
        L.b200pose_encode_persons_n.argtypes = [i32, vp, vp, vp, vp, vp, camp, vp, i32, vp, vp, i32, vp, vp]
        L.b200pose_split_planes.argtypes = [vp, i32, i32, i32, vp, vp, i32, vp]
        L.b200pose_gat_aggregate.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, f32, f32,
                                             vp, vp, vp, i32, vp, i32, vp]
        L.b200pose_gat_aggregate_res.argtypes = [i32, i32, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, f32, vp, i32,
                                                 vp, vp, vp, i32, vp, vp]
        L.b200pose_cluster.argtypes = [i32, vp, vp, vp, vp, vp, i32, f64, i32, i32, i32, vp, vp, vp]
        L.b200pose_cluster_pairs.argtypes = L.b200pose_cluster.argtypes
        L.b200pose_build_graph_pairs.argtypes = [i32, vp, vp, vp, camp, vp, i32, vp, vp, vp, vp, vp, vp]
        L.b200pose_encode_persons.argtypes = [i32, vp, vp, vp, vp, camp, vp, i32, vp, vp, i32, vp, vp]
        L.b200pose_triangulate.argtypes = [i32, vp, vp, vp, camp, i32, vp, vp, vp]
        L.b200pose_gather_persons.argtypes = [i32, vp, vp, vp, vp, i32, vp, i32, camp, vp, vp, vp]
        L.b200pose_pack_record.argtypes = [i32, i32, i32, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp]
        L.b200pose_pack_json.argtypes = [C.c_char_p, C.c_int64, i32, C.POINTER(C.c_char_p), C.POINTER(i32), i32, C.POINTER(vp)]
        L.b200pose_packed_sizes.argtypes = [vp] + [C.POINTER(i32)] * 5
        L.b200pose_packed_copy.argtypes = [vp] * 8 + [i32]
        L.b200pose_packed_free.argtypes = [vp]
        L.b200pose_packed_free.restype = None
        L.b200pose_gat_aggregate_bwd.argtypes = [i32, vp, vp, vp, i32, i32, i32, f32, vp, i32, vp, vp, vp, vp, i32, vp]
        L.b200pose_grad_planes.argtypes = [vp, i32, i32, i32, vp, i32, f32, vp, i32, vp, vp, i32, vp, vp, i32, vp]
        L.b200pose_transpose_planes.argtypes = [vp, vp, i32, i32, i32, vp, vp, i32, vp]
        L.b200pose_colsum.argtypes = [vp, i32, i32, i32, vp, i32, i32, vp, vp]
        L.b200pose_mse_sigmoid.argtypes = [vp, i32, vp, vp, i32, vp, vp, vp]
        L.b200pose_sigmoid_bwd.argtypes = [vp, vp, i32, vp, vp]
        L.b200pose_gat_prepare_layer.argtypes = [vp, vp, i32, vp, vp, vp, i32, i32, i32, vp, vp, i32, vp, vp, i32, vp, vp, i32, vp, vp, i32, vp, vp]
        L.b200pose_gat_attn_bias_grad.argtypes = [vp, i32, vp, i32, i32, i32, i32, vp, vp, vp, vp]
        L.b200pose_residual_bwd_add.argtypes = [vp, i32, vp, i32, i32, i32, i32, vp]
        L.b200pose_adam_step_dev.argtypes = [vp, vp, vp, vp, C.c_int64, f32, f32, f32, f32, f32, vp, vp, vp]
        L.b200pose_mlp_adam_planes.argtypes = [vp, vp, vp, vp, C.c_int64, C.POINTER(MlpLayer), i32, f32, f32, f32, f32, f32, vp, vp, vp]
        for name in EXPORTS:
            if name not in ('b200pose_last_error', 'b200pose_packed_free'):
                getattr(L, name).restype = C.c_int32
        _lib = L
    return _lib


def check(rc: int, what: str = ''):
    if rc != 0:
        msg = lib().b200pose_last_error()
        raise B200PoseError('%s failed (%d): %s' % (what or 'b200pose call', rc, (msg or b'').decode()))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())
