"""ctypes binding of libb200seg.so (declared in include/b200seg.h).

The library is a plain C ABI (raw device pointers + ints); this module is the only place that
touches it.  Loading never needs a GPU; calling any compute entry point without one fails inside
CUDA and surfaces as RuntimeError.  If the shared object is missing the import raises -- there is no
fallback implementation anywhere in the package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200seg.so")

F32, BF16 = 0, 1
I64, U8 = 2, 3              # target dtypes of the metrics entry points
NCHW, NHWC = 0, 1           # logits layouts of b200seg_seg_metrics
ACT_NONE, ACT_RELU, ACT_RELU6 = 0, 1, 2

_vp, _i, _f, _ll, _d = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_double

# name -> argtypes (restype is always int unless noted)
_PROTOS = {
    "b200seg_version": [],
    "b200seg_device_info": [C.POINTER(_i), C.POINTER(_i)],
    "b200seg_conv3x3_smallcin": [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_stem_mb1_supported": [_i, _i, _i, _i, _i],
    "b200seg_stem_mb1": [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp],
    "b200seg_dwconv3x3": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_dwconv3x3_bf16w": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_conv_tc": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_conv_rs_supported": [_i, _i, _i, _i],
    "b200seg_conv_rs": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_dwconv3x3_tc": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_mbconv": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_conv_simt": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_upsample2x_concat": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_upsample2x_ac_nchw": [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _vp],
    "b200seg_upsample2x_ac_argmax": [_vp, _i, _i, _vp, _i, _i, _i, _i, _vp],
    "b200seg_tail_fused": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp],
    "b200seg_tail_fused_metrics": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _ll, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "b200seg_seg_metrics": [_vp, _i, _i, _i, _vp, _i, _ll, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "b200seg_nhwc_to_nchw": [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _vp],
    "b200seg_maxpool2x2": [_vp, _vp, _i, _i, _i, _i, _i, _vp],
    "b200seg_softmax_ce": [_vp, _vp, _vp, _vp, _f, _vp, _i, _i, _i, _i, _vp],
    "b200seg_scale_unless_one": [_vp, _ll, _vp, _vp],
    "b200seg_remap_labels": [_vp, _vp, _vp, _ll, _vp],
    "b200seg_ce_count": [_vp, _vp, _ll, _i, _ll, _vp],
    "b200seg_softmax_ce_ex": [_vp, _vp, _i, _ll, _vp, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp],
    "b200seg_ce_count_ex": [_vp, _i, _ll, _vp, _vp, _ll, _i, _vp],
    "b200seg_softmax_ce_ex_bwd": [_vp, _vp, _i, _ll, _vp, _f, _vp, _vp, _i, _i, _i, _i, _vp],
    "b200seg_upsample2x_ac_generic": [_vp, _i, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp],
    "b200seg_final_bwd_generic": [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_nhwc_argmax": [_vp, _i, _i, _vp, _ll, _i, _vp],
    # training path
    "b200seg_bn_stats": [_vp, _i, _ll, _i, _vp, _vp, _i, _ll, _vp],
    "b200seg_bn_finalize": [_vp, _i, _vp, _vp, _i, _ll, _ll, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp],
    "b200seg_bn_apply": [_vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _i, _vp],
    "b200seg_bn_bwd_reduce": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _i, _vp, _vp, _i, _ll, _vp],
    "b200seg_bn_cluster_supported": [_i, _ll, _i],
    "b200seg_bn_cluster_bwd_supported": [_i, _ll, _i],
    "b200seg_bn_cluster_fwd": [_vp, _ll, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp, _i, _vp],
    "b200seg_bn_cluster_bwd": [_vp, _vp, _vp, _ll, _i, _i, _vp, _vp, _vp],
    "b200seg_bn_bwd_apply": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _i, _vp],
    "b200seg_bn_bwd_apply_slots": [_vp, _vp, _vp, _vp, _i, _vp, _i, _ll, _i, _i, _vp],
    "b200seg_bn_finalize_apply": [_vp, _vp, _i, _vp, _vp, _f, _f, _vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _i, _vp],
    "b200seg_act_bwd": [_vp, _vp, _vp, _i, _ll, _i, _vp],
    "b200seg_colsum": [_vp, _i, _ll, _i, _vp, _i, _ll, _vp],
    "b200seg_f64_to_f32": [_vp, _vp, _i, _i, _ll, _f, _vp],
    "b200seg_conv_wgrad": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_conv_wgrad_tc": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_dw_dgrad": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_dw_wgrad": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_smallcin_wgrad": [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_upcat_bwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_final_bwd": [_vp, _vp, _i, _i, _i, _i, _i, _vp],
    "b200seg_nchw_to_nhwc_pad": [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp],
    "b200seg_preprocess_u8": [_vp, _i, _i, _i, _vp, _i, _vp, _i, _i, _f, _f, _f, _f, _f, _f, _vp],
    "b200seg_adam_multi": [_vp, _vp, _vp, _i, _f, _d, _f, _d, _f, _f, _d, _d, _vp],
    "b200seg_adam_chunk": [],
    "b200seg_pack_weights_multi": [_vp, _vp, _vp, _i, _vp],
    "b200seg_pack_chunk": [],
    "b200seg_fold_pack_eval_multi": [_vp, _vp, _vp, _i, _vp],
    "b200seg_fold_chunk": [],
    "b200seg_grad_finalize_multi": [_vp, _vp, _vp, _i, _vp],
    "b200seg_grad_chunk": [],
    "b200seg_maxpool_bwd": [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp],
    # object boxes and overlay (postprocess.cu)
    "b200seg_detect_workspace_bytes": [_i, _i, _i, _i, C.POINTER(_ll)],
    "b200seg_detect_objects": [_vp, _i, _i, _i, _i, _i, C.POINTER(_i), _i, _i, _i, _i, _vp, _ll, _vp, _vp, _vp, _vp, _vp],
    "b200seg_overlay": [_vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _f, _f, _f, _vp, _vp],
}
EXPORTS = sorted(list(_PROTOS) + ["b200seg_last_error"])


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python team02-objectdetection_b200/build.py` "
            "(nvcc, sm_100a). b200seg has no CPU/eager fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, args in _PROTOS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = _i
    lib.b200seg_last_error.argtypes = []
    lib.b200seg_last_error.restype = C.c_char_p
    return lib


lib = _load()


LAUNCHES = [0]      # C-ABI calls that returned success (each is one kernel launch; two for a few wrappers' helpers)


def check(rc: int, what: str = "") -> None:
    LAUNCHES[0] += 1
    if rc != 0:
        msg = lib.b200seg_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"libb200seg {what} failed (rc={rc}): {msg}")


def ptr(t) -> int:
    """Raw device pointer of a torch tensor (None -> NULL)."""
    return 0 if t is None else t.data_ptr()


def device_info():
    sm, cc = _i(0), _i(0)
    check(lib.b200seg_device_info(C.byref(sm), C.byref(cc)), "device_info")
    return sm.value, cc.value
