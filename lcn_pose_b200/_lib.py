"""ctypes binding of liblcn_b200.so (include/lcn_b200.h).  Fails loudly when the library is missing."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LCN_B200_LIB: another build of the same library (the -DLCN_TC_PROFILE one, profiling scripts only)
LIB_PATH = os.path.abspath(os.environ.get("LCN_B200_LIB", os.path.join(_HERE, "liblcn_b200.so")))

J = 17
LCN_PATH_FP32, LCN_PATH_BF16 = 0, 1
LCN_MASK_LOCALLY_CONNECTED, LCN_MASK_CONSTANT = 0, 1
LCN_EVAL_PROTOCOL2, LCN_EVAL_CAMERA_FRAME = 1, 2
LCN_AUG_FLIP, LCN_AUG_ROTATE, LCN_AUG_TRANSLATE = 1, 2, 3


class LcnError(RuntimeError):
    pass


class ModelDesc(C.Structure):
    _fields_ = [("F", C.c_int32), ("in_F", C.c_int32), ("num_layers", C.c_int32), ("mask_kind", C.c_int32),
                ("residual", C.c_int32), ("batch_norm", C.c_int32), ("max_norm", C.c_int32), ("path", C.c_int32),
                ("support", C.c_float * (J * J)), ("const_mask", C.c_float * (J * J))]


# every exported symbol of include/lcn_b200.h with its prototype (restype, argtypes)
_vp, _i32, _i64, _u64, _f, _sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_size_t
PROTOTYPES = {
    "lcn_version": (C.c_char_p, []),
    "lcn_last_error": (C.c_char_p, []),
    "lcn_crc32c": (C.c_uint32, [_vp, _sz, C.c_uint32]),
    "lcn_neighbour_matrix": (C.c_int, [C.c_int, _vp]),
    "lcn_exponential_matrix": (C.c_int, [_vp]),
    "lcn_model_create": (C.c_int, [C.POINTER(ModelDesc), C.POINTER(_vp)]),
    "lcn_model_destroy": (None, [_vp]),
    "lcn_model_param_count": (_i64, [_vp]),
    "lcn_model_num_tensors": (C.c_int, [_vp]),
    "lcn_model_tensor_info": (C.c_int, [_vp, C.c_int, C.c_char_p, C.c_int, C.POINTER(_i64), C.POINTER(_i32), C.POINTER(_i32)]),
    "lcn_model_workspace_bytes": (_sz, [_vp, _i64, _i32, C.c_int]),
    "lcn_model_prepare_weights": (C.c_int, [_vp, _vp, _vp, _sz, _vp]),
    "lcn_model_forward": (C.c_int, [_vp, _vp, _vp, _sz, _vp, _i64, _i32, C.c_int, _f, _u64, _u64, _vp, _vp, _vp]),
    "lcn_model_forward_layers": (C.c_int, [_vp, _vp, _vp, _sz, _vp, _i64, _i32, _f, _u64, _u64, C.c_int, C.c_int, _vp, _vp]),
    "lcn_model_write_tensor": (C.c_int, [_vp, _vp, _sz, C.c_int, C.c_int, _i64, _i32, _vp, _vp]),
    "lcn_mask_weights": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _vp]),
    "lcn_batch_norm": (C.c_int, [_vp, _i64, _i32, _vp, _vp, _f, _vp, _vp, _vp]),
    "lcn_mse_loss": (C.c_int, [_vp, _vp, _i64, _vp, _f, _vp, _vp]),
    "lcn_l2_regularizer": (C.c_int, [_vp, _vp, _vp, _vp, _vp]),
    "lcn_loss_ema": (C.c_int, [_vp, _vp, _f, _f, _vp, _vp]),
    "lcn_gather_rows": (C.c_int, [_vp, _i32, _vp, _vp, _i32, _vp, _vp, _i64, _i64, _vp]),
    "lcn_normalize": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    "lcn_model_forward_taps": (C.c_int, [_vp, _vp, _vp, _sz, _vp, _i64, _i32, _vp, _vp, _sz, _vp]),
    "lcn_model_backward": (C.c_int, [_vp, _vp, _vp, _sz, _vp, _vp, _i64, _f, _u64, _u64, _vp, _vp, _vp]),
    "lcn_model_finalize_grads": (C.c_int, [_vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "lcn_model_grad_compact_count": (_i64, [_vp]),
    "lcn_model_pack_grads": (C.c_int, [_vp, _vp, _vp, _vp]),
    "lcn_model_unpack_grads": (C.c_int, [_vp, _vp, _vp, _vp]),
    "lcn_dp_export": (C.c_int, [_vp, C.c_int, _vp]),
    "lcn_dp_bucket": (_vp, [_vp]),
    "lcn_dp_connect": (C.c_int, [_vp, _vp, C.c_int, C.c_int]),
    "lcn_dp_world": (C.c_int, [_vp]),
    "lcn_dp_enable": (C.c_int, [_vp, C.c_int]),
    "lcn_dp_sync_batch_norm": (C.c_int, [_vp, C.c_int]),
    "lcn_model_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _sz, _vp, _f, _f, _f, _f, _f, _vp, _vp]),
    "lcn_layer_gemm": (C.c_int, [_vp, _vp, _vp, _sz, _i64, _i32, C.c_int, C.c_int, _vp]),
    "lcn_model_read_tensor": (C.c_int, [_vp, _vp, _sz, C.c_int, C.c_int, _i64, _i32, _vp, _vp]),
    "lcn_dropout_mask": (C.c_int, [_u64, _u64, C.c_int, _i64, _i32, _f, _vp, _vp]),
    "lcn_eval_mpjpe": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, C.c_int, _vp, _vp, _vp, _vp]),
    "lcn_procrustes": (C.c_int, [_vp, _vp, _i64, C.c_int, C.c_int, _vp, _vp, _vp]),
    "lcn_denormalize": (C.c_int, [_vp, _vp, _i64, _vp]),
    "lcn_augment": (C.c_int, [_vp, _vp, _i64, C.c_int, C.c_int, _f, _f, _vp]),
    "lcn_tta_undo": (C.c_int, [_vp, _vp, _i64, C.c_int, C.c_int, C.c_int, C.c_int, _f, _f, _vp]),
}

_lib = None


def load():
    """Load liblcn_b200.so.  No fallback: a missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LcnError(f"{LIB_PATH} not found: build it with `python __graft_entry__.py build` "
                       f"(make -C lcn_pose_b200/csrc). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise LcnError(f"liblcn_b200 error {rc}: {load().lcn_last_error().decode()}")


def neighbour_matrix(knn):
    import numpy as np
    out = np.zeros((J, J), dtype=np.float32)
    check(load().lcn_neighbour_matrix(int(knn), out.ctypes.data))
    return out


def exponential_matrix():
    import numpy as np
    out = np.zeros((J, J), dtype=np.float32)
    check(load().lcn_exponential_matrix(out.ctypes.data))
    return out
