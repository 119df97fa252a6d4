"""ctypes binding of libsketchedit_b200.so (include/sketchedit_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, the
caller gets an exception. Loading the library does not need a GPU (symbol checks run on CPU);
running anything does.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SE_B200_LIB") or os.path.join(_HERE, "libsketchedit_b200.so")   # SE_B200_LIB: an A/B build of the same sources

_c_void_p = ctypes.c_void_p
_c_int = ctypes.c_int
_c_char = ctypes.c_char
_c_char_p = ctypes.c_char_p
_fp = ctypes.POINTER(ctypes.c_float)

# name -> (restype, argtypes); must list every symbol include/sketchedit_b200.h declares
SIGNATURES = {
    "se_last_error": (_c_char_p, []),
    "se_abi_version": (_c_int, []),
    "se_model_create": (_c_int, [ctypes.POINTER(_c_void_p)]),
    "se_model_destroy": (None, [_c_void_p]),
    "se_model_set_layer": (_c_int, [_c_void_p, _c_char, _c_char_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int]),
    "se_model_finalize": (_c_int, [_c_void_p]),
    "se_model_set_option": (_c_int, [_c_void_p, _c_int, _c_int]),
    "se_forward_inference": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int,
                                      _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p,
                                      _c_void_p]),
    "se_forward_inference_packed": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_void_p, _c_void_p]),
    "se_forward_inference_u8": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_void_p, _c_void_p, _c_void_p]),
    "se_forward_inpaint": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_void_p, _c_void_p,
                                    _c_void_p, _c_void_p]),
    "se_forward_inpaint_u8": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_void_p, _c_void_p]),
    "se_netM_forward": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_void_p, _c_void_p,
                                 _c_void_p]),
    "se_netG_forward": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_int,
                                 _c_int, _c_void_p, _c_void_p, _c_void_p]),
    "se_gated_conv_forward": (_c_int, [_c_void_p, _c_char, _c_char_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_void_p,
                                       _c_void_p]),
    "se_contextual_attention_forward": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_int, _c_int, _c_void_p,
                                                 _c_void_p, _c_void_p]),
    "se_outputs_to_uint8": (_c_int, [_c_void_p, _c_void_p, _c_int, _c_int, _c_int, _c_void_p, _c_void_p, _c_void_p]),
    "se_resize_u8": (_c_int, [_c_void_p, _c_void_p, _c_void_p, _c_int, _c_int, _c_void_p, _c_void_p, _c_void_p, _c_int, _c_void_p]),
    "se_resize_coeffs": (_c_int, [_c_int, _c_int, _c_void_p, _c_void_p, _c_int]),
    "se_last_launch_count": (_c_int, []),
    "se_workspace_bytes": (ctypes.c_longlong, [_c_void_p]),
    "se_timing_enable": (_c_int, [_c_int]),
    "se_timing_report": (_c_int, [_c_char_p, _c_int]),
}

_lib = None


class SketchEditB200Error(RuntimeError):
    pass


def load():
    """Load the library (building nothing: run `python -m sketchedit_b200.build` first)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SketchEditB200Error(
            "%s not found. Build it with `python -m sketchedit_b200.build` (nvcc, sm_100a). "
            "There is no CPU or PyTorch fallback for this path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().se_last_error()
        raise SketchEditB200Error("sketchedit_b200 call failed (rc=%d): %s" % (rc, msg.decode() if msg else "?"))


# "fp32": fp32-parity arithmetic on the tensor cores (split-half fp16, SE_PREC_FP32_TC); "fp32_direct": the fp32 CUDA-core kernels
PREC = {"bf16": 0, "fp32": 3, "fp32_direct": 1, "bf16_direct": 2}
RESIZE_REVERSE_CHANNELS = 1   # SE_RESIZE_REVERSE_CHANNELS
OPT = {"use_cam": 0, "pool_avg": 1, "no_mask_cc": 2, "no_mask_coarse": 3, "joint_train_inp": 4}
