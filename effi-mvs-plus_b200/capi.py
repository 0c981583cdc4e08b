"""ctypes binding of libeffimvs.so (include/effimvs.h).  No torch types cross this boundary:
only raw device pointers, sizes and a cudaStream_t.  Importing this module raises if the
library has not been built (``python -c "import __graft_entry__ as g; g.build()"`` or
``make -C effi-mvs-plus_b200/csrc``) -- there is no CPU or eager fallback."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("EFFIMVS_LIB") or os.path.join(_HERE, "libeffimvs.so")   # EFFIMVS_LIB: kernel-tuning builds

OK, EINVAL, EUNSUPPORTED, ECUDA, EWORKSPACE = 0, -1, -2, -3, -4
HYP_TENSOR, HYP_PLANES, HYP_LOCAL = 0, 1, 2
RANGE_SCALAR, RANGE_PIXEL = 0, 1
FEA_NCHW, FEA_NHWC = 0, 1
PREC_F32, PREC_BF16, PREC_BF16X3 = 0, 1, 2
WS_PREPARE, WS_RUN = 1, 2
CONV2D_BIAS, CONV2D_BIAS_RELU, CONV2D_ADD_RELU, CONV2D_GRU_GATES, CONV2D_GRU_UPDATE = 0, 1, 2, 3, 4
MAX_SRC_VIEWS = 16


class EffiMVSError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libeffimvs error {}: {}".format(code, msg))
        self.code = code


if not os.path.exists(LIB_PATH):
    raise ImportError("libeffimvs.so is not built ({}); run __graft_entry__.build() -- the hot path has no "
                      "CPU or PyTorch fallback".format(LIB_PATH))

lib = C.CDLL(LIB_PATH)

_p, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
_pp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); mirrors include/effimvs.h one to one
SIGNATURES = {
    "effimvs_last_error": (C.c_char_p, []),
    "effimvs_version": (_i, []),
    "effimvs_relative_projection_f32": (_i, [_p, _i, _i, _p, _p]),
    "effimvs_homo_warp_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "effimvs_depth_range_samples_f32": (_i, [_p, _p, _i, _i, _i, _i, _p, _p]),
    "effimvs_depth_ranges_f32": (_i, [_p, _i, _i, _i, _p, _p, _p]),
    "effimvs_fusion_masks_f32": (_i, [_p, _p, _i, _i, _i, _i, _f, _f, _i, _i, _p, _p]),
    "effimvs_warp_corr_agg_f32": (_i, [_p, _pp, _i, _p, _p, _i, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p]),
    "effimvs_warp_corr_views_f32": (_i, [_p, _pp, _i, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p, _p]),
    "effimvs_weighted_agg_f32": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "effimvs_volume_lookup_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _p, _p]),
    "effimvs_dynamic_cost_f32": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p]),
    "effimvs_softmax_regress_conf_f32": (_i, [_p, _p, _i, _i, _i, _i, _i, _p, _p, _p]),
    "effimvs_conv3d_f32": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _i, _i, _p]),
    "effimvs_conv3d_bf16_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i, _i, _i]),
    "effimvs_conv3d_bf16": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _p, _sz, _p, _p]),
    "effimvs_costreg_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "effimvs_costreg_fpn3d": (_i, [_p, _pp, _pp, _i, _i, _i, _i, _i, _p, _sz, _p, _p]),
    "effimvs_cost_up_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "effimvs_cost_up_small": (_i, [_p, _p, _pp, _pp, _i, _i, _i, _i, _i, _p, _sz, _p, _p]),
    "effimvs_costreg_fpn3d_ex": (_i, [_p, _pp, _pp, _i, _i, _i, _i, _i, _i, _p, _sz, _p, _p]),
    "effimvs_cost_up_small_ex": (_i, [_p, _p, _pp, _pp, _i, _i, _i, _i, _i, _i, _p, _sz, _p, _p]),
    "effimvs_gru_reset_f32": (_i, [_p, _p, _p, C.c_longlong, _i, _i, _p, _p]),
    "effimvs_gru_update_f32": (_i, [_p, _p, _p, _p, _p, C.c_longlong, _i, _i, _p, _p]),
    "effimvs_gru_delta_f32": (_i, [_p, _p, _p, _p, _p, _i, _i, _p, _p, _p]),
    "effimvs_inv_init_f32": (_i, [_p, _p, _p, _i, _i, _p, _p, _p]),
    "effimvs_delta_head_f32": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "effimvs_convex_upsample_f32": (_i, [_p, _p, _f, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "effimvs_convex_upsample_conv_f32": (_i, [_p, _i, _p, _p, _f, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "effimvs_encoder_head_f32": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "effimvs_encoder_head_hostw_f32": (_i, [_p, _p, _p, _i, _i, _i, _i, _i, _p, _p]),
    "effimvs_encoder_head_pack_host": (_i, [_p, _p, _p, _p, _i, _i, _p]),
    "effimvs_encoder_head_table_floats": (_i, [_i]),
    "effimvs_encoder_tail_f32": (_i, [_p, _p, _p, C.c_longlong, _i, _i, _p, _p]),
    "effimvs_encoder_tail_ctx_f32": (_i, [_p, _p, _p, _i, _i, _i, _p, _p, C.c_longlong, _i, _i, _p, _p]),
    "effimvs_conv2d_tf32_supported": (_i, [_i, _i]),
    "effimvs_conv2d_tf32_packed_bytes": (_sz, [_i, _i]),
    "effimvs_conv2d_tf32_pack": (_i, [_p, _i, _i, _p, _p]),
    "effimvs_conv2d_bf16x3_supported": (_i, [_i, _i]),
    "effimvs_conv2d_bf16x3_packed_bytes": (_sz, [_i, _i]),
    "effimvs_conv2d_bf16x3_pack": (_i, [_p, _i, _i, _p, _p]),
    "effimvs_conv2d_bf16x3": (_i, [_p, C.c_longlong, _i, _p, C.c_longlong, _i, _p, _p, _i, _i, _i, _i, _i,
                                   _p, C.c_longlong, _p, C.c_longlong, _p, C.c_longlong, _p]),
    "effimvs_conv2d_tf32": (_i, [_p, C.c_longlong, _i, _p, C.c_longlong, _i, _p, _p, _i, _i, _i, _i, _i,
                                 _p, C.c_longlong, _p, C.c_longlong, _p, C.c_longlong, _p]),
    "effimvs_gru_init_f32": (_i, [_p, C.c_longlong, _i, _i, _p, _p]),
    "effimvs_gru_init_ctx_f32": (_i, [_p, C.c_longlong, _i, _i, _p, _p, _p, _p, _p]),
    "effimvs_dtu_filter_f32": (_i, [_p, _p, _p, _p, C.POINTER(C.c_double), C.POINTER(C.c_float), _i, _i, _i, _f, _f, _i, _i, _i,
                                    _p, _p, _p, _p, _p, _p, _p]),
    "effimvs_dtu_filter_views_f32": (_i, [_p, _i, _p, _p, _p, _i, _p, _p, C.POINTER(C.c_double), C.POINTER(C.c_float), _i, _i, _i,
                                          _f, _f, _i, _i, _i, _p, _p, _p, _p, _p]),
    "effimvs_images_u8_to_f32": (_i, [_p, C.c_longlong, _p, _p]),
    "effimvs_fusion_invert_cameras_f32": (_i, [_p, _p, _i, _i, _p, _p]),
    "effimvs_fusion_reproject_f32": (_i, [_p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _p]),
    "effimvs_fusion_filter_f32": (_i, [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _f, _f, _i, _f, _i, _p, _p, _p, _p, _p]),
    "effimvs_fusion_filter_views_f32": (_i, [_p, _i, _p, _p, _p, _i, _p, _p, _p, _i, _i, _f, _f, _i, _f, _i, _i, _i, _i,
                                             _p, _p, _p, _p]),
    "effimvs_point_offsets_workspace_bytes": (_sz, [_i, _i, _i]),
    "effimvs_point_offsets": (_i, [_p, _i, _i, _i, _p, _sz, _p, _p]),
    "effimvs_gather_points_f32": (_i, [_p, _p, _p, _i, _p, _i, _i, _i, _p, _sz, _p, _p, _p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)        # AttributeError here = header and library disagree
    _fn.restype = _res
    _fn.argtypes = _args


def last_error() -> str:
    return lib.effimvs_last_error().decode("utf-8", "replace")


def check(rc: int) -> None:
    if rc != OK:
        raise EffiMVSError(rc, last_error())


def ptr_array(ptrs):
    """Host array of device pointers (``const float* const*``)."""
    arr = (C.c_void_p * len(ptrs))(*[C.c_void_p(p) for p in ptrs])
    return C.cast(arr, _pp), arr     # keep `arr` alive for the duration of the call
