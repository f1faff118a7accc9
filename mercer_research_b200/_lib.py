"""ctypes binding of librcn_cuda.so -- the C ABI declared in include/rcn_cuda.h.

This is the ONLY compute backend of the package: if the shared library is missing, or no CUDA device is
usable, calls raise. There is no CPU fallback and nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("RCN_CUDA_LIB") or os.path.join(_HERE, "librcn_cuda.so")   # env override: A/B-testing a build

RCN_OK = 0
STATUS_NAMES = {
    0: "RCN_OK", 1: "RCN_ERR_INVALID", 2: "RCN_ERR_SHAPE", 3: "RCN_ERR_NOT_IMPLEMENTED", 4: "RCN_ERR_CUDA",
    5: "RCN_ERR_STATE", 6: "RCN_ERR_OUT_OF_BOUNDS", 7: "RCN_ERR_NAN",
}

PIXELS_U8_ROWMAJOR = 0
PIXELS_F64_COLMAJOR = 1
PIXELS_F64_NHWC = 2

# name -> argtypes; every function returns int (rcn_status) unless listed in _RESTYPES.
_vp, _sz, _i, _d = C.c_void_p, C.c_size_t, C.c_int, C.c_double
_szp = C.POINTER(C.c_size_t)
SIGNATURES = {
    "rcn_cuda_version": [],
    "rcn_cuda_device_count": [C.POINTER(C.c_int)],
    "rcn_cuda_create": [_sz, _vp, _sz, _vp, _sz, _i, C.POINTER(_vp)],
    "rcn_cuda_destroy": [_vp],
    "rcn_cuda_set_stream": [_vp, _vp],
    "rcn_cuda_synchronize": [_vp],
    "rcn_cuda_feature_shape": [_vp, _sz, _sz, _szp, _szp, _szp],
    "rcn_cuda_init_params": [_vp, _sz],
    "rcn_cuda_init_params_shapes": [_vp, _vp, _vp, _sz],
    "rcn_cuda_num_layers": [_vp, _szp],
    "rcn_cuda_layer_shape": [_vp, _sz, _szp, _szp],
    "rcn_cuda_param_count": [_vp, _szp],
    "rcn_cuda_set_weights": [_vp, _sz, _sz, _sz, _vp],
    "rcn_cuda_get_weights": [_vp, _sz, _vp],
    "rcn_cuda_set_bias": [_vp, _sz, _sz, _vp],
    "rcn_cuda_get_bias": [_vp, _sz, _vp],
    "rcn_cuda_set_params": [_vp, _vp, _sz],
    "rcn_cuda_get_params": [_vp, _vp, _sz],
    "rcn_cuda_set_scale": [_vp, _d, _d],
    "rcn_cuda_get_scale": [_vp, C.POINTER(_d), C.POINTER(_d)],
    "rcn_cuda_features": [_vp, _vp, _i, _sz, _sz, _sz, _i, _vp],
    "rcn_cuda_gen_scales": [_vp, _vp, _sz, _sz, C.POINTER(_d), C.POINTER(_d)],
    "rcn_cuda_standardise": [_vp, _vp, _sz],
    "rcn_cuda_forward": [_vp, _vp, _sz, _vp],
    "rcn_cuda_classify_features": [_vp, _vp, _sz, _vp],
    "rcn_cuda_classify": [_vp, _vp, _i, _sz, _sz, _sz, _vp],
    "rcn_cuda_evaluate": [_vp, _vp, _vp, _sz, C.POINTER(C.c_uint64)],
    "rcn_cuda_evaluate_images": [_vp, _vp, _i, _vp, _sz, _sz, _sz, _vp, _vp, _vp],
    "rcn_cuda_accumulate_gradients": [_vp, _vp, _vp, _vp, _sz],
    "rcn_cuda_accumulate_gradients_images": [_vp, _vp, _i, _vp, _sz, _sz, _sz],
    "rcn_cuda_apply_gradients": [_vp, _d, _sz],
    "rcn_cuda_train_batch": [_vp, _vp, _vp, _vp, _sz, _d],
    "rcn_cuda_train_batch_images": [_vp, _vp, _i, _vp, _sz, _sz, _sz, _d],
    "rcn_cuda_last_batch_stats": [_vp, C.POINTER(_d), C.POINTER(C.c_uint64)],
    "rcn_cuda_epoch_bind": [_vp, _vp, _i, _vp, _vp, _sz, _sz, _sz, _sz],
    "rcn_cuda_epoch_seek": [_vp, _sz],
    "rcn_cuda_epoch_position": [_vp, _szp],
    "rcn_cuda_epoch_accumulate": [_vp],
    "rcn_cuda_epoch_apply": [_vp, _d, _sz],
    "rcn_cuda_epoch_step": [_vp, _d],
    "rcn_cuda_epoch_run": [_vp, _d, _sz],
    "rcn_cuda_train_epoch_host": [_vp, _vp, _i, _vp, _sz, _sz, _sz, _sz, _d, _sz, _vp, _vp, _szp],
    "rcn_cuda_dp_init": [_vp, _i, _i, _vp],
    "rcn_cuda_dp_connect_ipc": [_vp, _vp],
    "rcn_cuda_dp_connect_local": [_vp, _vp],
    "rcn_cuda_dp_shutdown": [_vp],
    "rcn_cuda_dp_error": [_vp, _vp],
    "rcn_cuda_timeline_enable": [_vp, _i],
    "rcn_cuda_timeline_read": [_vp, _vp, _vp],
    "rcn_cuda_bind_gradient_buffer": [_vp, _vp, _sz],
    "rcn_cuda_gradient_buffer": [_vp, C.POINTER(_vp), _szp],
    "rcn_cuda_get_gradients": [_vp, _vp, _sz],
    "rcn_cuda_get_activations": [_vp, _sz, _vp],
    "rcn_cuda_get_deltas": [_vp, _sz, _vp],
    "rcn_cuda_kernel_launches": [C.POINTER(C.c_uint64)],
    "rcn_cuda_allocation_generation": [C.POINTER(C.c_uint64)],
    "rcn_cuda_profile_enable": [_i],
    "rcn_cuda_profile_report": [C.c_char_p, _sz],
    "rcn_cuda_convolve_2d": [_i, _vp, _vp, _sz, _sz, _vp, _sz, _sz, _i, _vp],
    "rcn_cuda_convolve_2d_separated": [_i, _vp, _vp, _sz, _sz, _i, _i, _vp],
    "rcn_cuda_relu": [_i, _vp, _vp, _sz, _vp],
    "rcn_cuda_pool_2d": [_i, _vp, _vp, _sz, _sz, _i, _i, _vp, _vp],
    # extensions (not in the reference; SURVEY.md 8a x1-x3)
    "rcn_cuda_ext_conv2d_forward": [_i, _vp, _vp, _sz, _sz, _sz, _sz, _vp, _vp, _sz, _sz, _sz, _i, _i, _vp],
    "rcn_cuda_ext_activation_backward": [_i, _vp, _vp, _vp, _sz, _i, _vp],
    "rcn_cuda_ext_conv2d_backward_data": [_i, _vp, _vp, _sz, _sz, _sz, _sz, _vp, _sz, _sz, _sz, _i, _vp, _i, _vp],
    "rcn_cuda_ext_conv2d_backward_weight": [_i, _vp, _vp, _vp, _sz, _sz, _sz, _sz, _sz, _sz, _sz, _i, _vp, _vp],
    "rcn_cuda_ext_pool2d_forward": [_i, _vp, _vp, _sz, _sz, _sz, _sz, _i, _i, _vp, _vp],
    "rcn_cuda_ext_pool2d_backward": [_i, _vp, _vp, _vp, _sz, _sz, _sz, _sz, _i, _i, _vp],
    "rcn_cuda_ext_softmax_xent": [_i, _vp, _vp, _sz, _sz, _vp, _vp, _vp, _vp, _vp],
    "rcn_cuda_ext_gemm_f64": [_i, _vp, _vp, _sz, _i, _vp, _sz, _i, _sz, _sz, _sz, _i, _vp],
    # convolutional network handle (learned conv / pool layers + the dense stack)
    "rcn_cuda_cnn_create": [_i, _sz, _sz, _sz, _vp, _sz, _vp, _sz, _sz, C.POINTER(_vp)],
    "rcn_cuda_cnn_create_with_head": [_i, _sz, _sz, _sz, _vp, _sz, _vp, _sz, _sz, _i, C.POINTER(_vp)],
    "rcn_cuda_cnn_destroy": [_vp],
    "rcn_cuda_cnn_set_stream": [_vp, _vp],
    "rcn_cuda_cnn_synchronize": [_vp],
    "rcn_cuda_cnn_layer_shape": [_vp, _sz, _szp, _szp, _szp],
    "rcn_cuda_cnn_param_count": [_vp, _szp],
    "rcn_cuda_cnn_set_params": [_vp, _vp, _sz],
    "rcn_cuda_cnn_get_params": [_vp, _vp, _sz],
    "rcn_cuda_cnn_accumulate": [_vp, _vp, _i, _vp, _sz, _sz, _sz],
    "rcn_cuda_cnn_apply": [_vp, _d, _sz],
    "rcn_cuda_cnn_train_batch": [_vp, _vp, _i, _vp, _sz, _sz, _sz, _d],
    "rcn_cuda_cnn_last_batch_stats": [_vp, C.POINTER(_d), C.POINTER(C.c_uint64)],
    "rcn_cuda_cnn_epoch_bind": [_vp, _vp, _i, _vp, _vp, _sz, _sz, _sz, _sz],
    "rcn_cuda_cnn_epoch_seek": [_vp, _sz],
    "rcn_cuda_cnn_epoch_position": [_vp, _szp],
    "rcn_cuda_cnn_epoch_accumulate": [_vp],
    "rcn_cuda_cnn_epoch_apply": [_vp, _d, _sz],
    "rcn_cuda_cnn_epoch_step": [_vp, _d],
    "rcn_cuda_cnn_epoch_run": [_vp, _d, _sz],
    "rcn_cuda_cnn_evaluate_images": [_vp, _vp, _i, _vp, _sz, _sz, _sz, _vp, _vp, _vp],
    "rcn_cuda_cnn_classify_images": [_vp, _vp, _i, _sz, _sz, _sz, _vp],
    "rcn_cuda_cnn_bind_gradient_buffer": [_vp, _vp, _sz],
    "rcn_cuda_cnn_gradient_buffer": [_vp, C.POINTER(_vp), _szp],
    "rcn_cuda_cnn_get_gradients": [_vp, _vp, _sz],
    "rcn_cuda_cnn_get_layer_output": [_vp, _sz, _vp],
    "rcn_cuda_cnn_get_input_gradient": [_vp, _vp],
    "rcn_cuda_cnn_set_optimizer": [_vp, _i, _d, _i, _d, _d, _d, _d],
    "rcn_cuda_cnn_optimizer_state_size": [_vp, _szp],
    "rcn_cuda_cnn_get_optimizer_state": [_vp, _vp, _sz],
    "rcn_cuda_cnn_set_optimizer_state": [_vp, _vp, _sz],
}
_RESTYPES = {"rcn_cuda_last_error": C.c_char_p}


class RcnCudaError(RuntimeError):
    """A librcn_cuda call failed. ``status`` is the rcn_status code; where the reference would panic!()
    the message is the reference's panic message."""

    def __init__(self, status: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")
        self.status = status
        self.message = message


_lib = None


def load() -> C.CDLL:
    """Loads librcn_cuda.so (built in-tree by __graft_entry__.build() / csrc/Makefile). Fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError(
            f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). mercer_research_b200 has no CPU fallback.")
    lib = C.CDLL(SO_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.rcn_cuda_last_error.argtypes = []
    lib.rcn_cuda_last_error.restype = C.c_char_p
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != RCN_OK:
        msg = load().rcn_cuda_last_error()
        raise RcnCudaError(status, msg.decode("utf-8", "replace") if msg else "")


def kernel_launches() -> int:
    """Kernels launched by librcn_cuda in this process (bench.py's gpu_launches)."""
    n = C.c_uint64()
    check(load().rcn_cuda_kernel_launches(C.byref(n)))
    return n.value


def allocation_generation() -> int:
    """Changes whenever the library (re)allocates one of its device buffers: a captured CUDA graph of library calls is
    only valid while this value is the one seen at capture time."""
    n = C.c_uint64()
    check(load().rcn_cuda_allocation_generation(C.byref(n)))
    return n.value


def profile_enable(on: bool) -> None:
    check(load().rcn_cuda_profile_enable(1 if on else 0))


def profile_report() -> dict:
    import json
    buf = C.create_string_buffer(1 << 16)
    check(load().rcn_cuda_profile_report(buf, len(buf)))
    return json.loads(buf.value.decode())
