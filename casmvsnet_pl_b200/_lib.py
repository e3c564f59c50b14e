"""ctypes binding of libcasmvs.so (C ABI declared in include/casmvs.h).

There is deliberately no fallback: if the shared library is missing or the
device is not a B200-class GPU the import / call fails loudly.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_size_t, c_uint64, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcasmvs.so")

NCHW, NHWC = 0, 1
ROUND_TF32 = 256
KEEP_FP32_OUT = 256      # OR-ed into conv3d precision
FP32, TF32 = 0, 1
CONV, CONV_TRANSPOSE, CONV_PLANAR = 0, 1, 2
PRECISIONS = {"fp32": FP32, "tf32": TF32}

# name -> (restype, argtypes); must list every symbol include/casmvs.h declares
SIGNATURES = {
    "casmvs_version": (c_int, []),
    "casmvs_last_error": (c_char_p, []),
    "casmvs_device_check": (c_int, [c_int]),
    "casmvs_launch_count": (c_uint64, []),
    "casmvs_fallback_count": (c_uint64, []),
    "casmvs_release_weight_images": (c_int, [c_void_p, c_size_t]),
    "casmvs_weight_cache_generation": (c_uint64, []),
    "casmvs_weight_image_count": (c_int, [c_void_p, c_size_t]),
    "casmvs_settle_weight_images": (c_int, []),
    "casmvs_warp_cost_workspace_bytes": (c_size_t, [c_int] * 6),
    "casmvs_warp_cost_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                     c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p, c_size_t, c_void_p]),
    "casmvs_homo_warp_fwd": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                     c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "casmvs_packed_conv3d_weight_floats": (c_size_t, [c_int, c_int]),
    "casmvs_pack_conv3d_weights": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "casmvs_invalidate_weight_cache": (c_int, []),
    "casmvs_conv3d_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p,
                                  c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                  c_int, c_int, c_int, c_void_p]),
    "casmvs_costreg_param_floats": (c_size_t, [c_int]),
    "casmvs_costreg_layer_info": (c_int, [c_int, c_int, POINTER(c_int), POINTER(c_int),
                                          POINTER(c_int), POINTER(c_int), POINTER(c_size_t),
                                          POINTER(c_size_t), POINTER(c_size_t)]),
    "casmvs_costreg_workspace_bytes": (c_size_t, [c_int] * 5),
    "casmvs_costreg_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "casmvs_regress_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "casmvs_depth_hypotheses_fwd": (c_int, [c_void_p, c_int, c_float, c_float, c_void_p,
                                            c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "casmvs_uniform_hypotheses_fwd": (c_int, [c_float, c_float, c_void_p, c_void_p, c_void_p,
                                              c_int, c_int, c_int, c_int, c_void_p]),
    "casmvs_depth_first_fwd": (c_int, [c_void_p, c_int, c_float, c_float, c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_void_p]),
    "casmvs_warp_cost_ladder_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p,
                                            c_float, c_void_p] + [c_int] * 8 + [c_void_p]),
    "casmvs_regress_ladder_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_float,
                                          c_void_p, c_void_p, c_void_p] + [c_int] * 4 + [c_void_p]),
    "casmvs_fpn_level_fwd": (c_int, [c_void_p] * 8 + [c_int] * 5 + [c_void_p]),
    "casmvs_fpn_merge_fwd": (c_int, [c_void_p] * 5 + [c_int] * 5 + [c_void_p]),
    "casmvs_conv2d_rgb8_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p] + [c_int] * 4 + [c_void_p]),
    "casmvs_conv2d_5x5s2_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p] + [c_int] * 6 + [c_void_p]),
    "casmvs_conv2d_5x5s2_fp32_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_void_p] + [c_int] * 5 + [c_void_p]),
    "casmvs_bias_act_nhwc": (c_int, [c_void_p, c_void_p, c_float, c_size_t, c_int, c_int, c_void_p]),
    "casmvs_bias_lrelu_nhwc": (c_int, [c_void_p, c_void_p, c_float, c_size_t, c_int, c_void_p]),
    "casmvs_normalize_u8_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(c_float),
                                        POINTER(c_float), c_void_p]),
    "casmvs_resize_u8_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                     c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                     c_void_p]),
    "casmvs_warp_cost_bwd": (c_int, [c_void_p] * 5 + [c_int] * 7 + [c_void_p]),
    "casmvs_conv3d_wgrad": (c_int, [c_void_p] * 3 + [c_int] * 10 + [c_void_p]),
    "casmvs_regress_bwd": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p] + [c_int] * 4 + [c_void_p]),
    "casmvs_geo_fuse_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                    POINTER(c_float), POINTER(c_float), c_void_p, c_int, c_int,
                                    c_int, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "casmvs_nchw_to_nhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_size_t, c_void_p]),
    "casmvs_nhwc_to_nchw": (c_int, [c_void_p, c_void_p, c_int, c_int, c_size_t, c_void_p]),
}

_lib = None


class CasMVSError(RuntimeError):
    pass


def load():
    """Load libcasmvs.so (once) and bind every symbol of the header."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise CasMVSError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (or `make -C casmvsnet_pl_b200/csrc`). There is no CPU/PyTorch "
            "fallback for the hot path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().casmvs_last_error()
        raise CasMVSError(f"{what}: {msg.decode() if msg else 'error'} (status {rc})")


def launch_count():
    return int(load().casmvs_launch_count())


def fallback_count():
    """tf32-mode layers that ran on the CUDA-core kernel because no tcgen05 kernel covers
    their shape (0 for the reference architecture)."""
    return int(load().casmvs_fallback_count())


def weight_cache_generation():
    return int(load().casmvs_weight_cache_generation())
