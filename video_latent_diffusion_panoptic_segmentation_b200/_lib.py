"""ctypes binding of libldmseg_b200.so (the C ABI declared in include/ldmseg_b200.h).

There is no CPU fallback: if the shared library is missing, or the device is not an sm_100 part, every compute
entry point raises. ``load()`` only dlopens the library (works without a GPU, used by the CPU symbol test).
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libldmseg_b200.so")

c_i32, c_i64, c_f32, c_f64, c_vp = C.c_int32, C.c_int64, C.c_float, C.c_double, C.c_void_p

LDM_GEMM_OUT_F32 = 1 << 0
LDM_GEMM_GEGLU = 1 << 1
LDM_GEMM_QKV_SPLIT = 1 << 2
LDM_GEMM_SILU = 1 << 3
LDM_GEMM_CONVT_LN_SILU = 1 << 4
LDM_GEMM_OUT_NCHW_F32 = 1 << 5

HASH_EMPTY = 0x8000000000000000
ABI_VERSION = 4  # must equal ldm_abi_version() of the built library (descriptor struct layouts)


class GemmDesc(C.Structure):
    _fields_ = [
        ("a1", c_vp), ("a2", c_vp), ("w", c_vp), ("bias", c_vp), ("rowbias", c_vp), ("residual", c_vp),
        ("out", c_vp), ("q", c_vp), ("k", c_vp), ("vt", c_vp), ("ln_gamma", c_vp), ("ln_beta", c_vp),
        ("ln_eps", c_f32),
        ("B", c_i32), ("H", c_i32), ("W", c_i32), ("c1", c_i32), ("c2", c_i32), ("N", c_i32), ("taps", c_i32),
        ("block_n", c_i32), ("flags", c_i32),
        ("heads", c_i32), ("head_dim", c_i32), ("dpad", c_i32), ("seq", c_i32), ("seq_pad", c_i32),
        ("vt_rows", c_i32), ("n_store", c_i32), ("qkv_part0", c_i32),
        ("identity", c_vp), ("splitk_ws", c_vp), ("splitk_ws_bytes", C.c_int64),
        ("row_stats_out", c_vp), ("ln_stats", c_vp), ("ln_colsum", c_vp), ("ln_fold_eps", c_f32), ("ln_parts", c_i32),
        ("a_stride", c_i32), ("a_pad", c_i32), ("a_H", c_i32), ("a_W", c_i32),
        ("up2", c_i32), ("out_H", c_i32), ("out_W", c_i32),
    ]


class AttnDesc(C.Structure):
    _fields_ = [
        ("q", c_vp), ("k", c_vp), ("vt", c_vp), ("out", c_vp),
        ("B", c_i32), ("heads", c_i32), ("seq", c_i32), ("head_dim", c_i32), ("dpad", c_i32), ("seq_pad", c_i32),
        ("vt_rows", c_i32), ("scale", c_f32), ("kv_seq", c_i32),
    ]


class GroupNormDesc(C.Structure):
    _fields_ = [
        ("x1", c_vp), ("x2", c_vp), ("gamma", c_vp), ("beta", c_vp), ("out", c_vp), ("stats", c_vp),
        ("B", c_i32), ("HW", c_i32), ("c1", c_i32), ("c2", c_i32), ("groups", c_i32), ("eps", c_f32), ("silu", c_i32),
    ]


# name -> (restype, argtypes); must list every symbol include/ldmseg_b200.h declares (tests/test_abi.py checks)
SIGNATURES = {
    "ldm_abi_version": (C.c_int, []),
    "ldm_last_error": (C.c_char_p, []),
    "ldm_check_device": (C.c_int, []),
    "ldm_launch_count": (C.c_longlong, []),
    "ldm_gemm_bf16": (C.c_int, [C.POINTER(GemmDesc), c_vp]),
    "ldm_flash_attn_fwd": (C.c_int, [C.POINTER(AttnDesc), c_vp]),
    "ldm_attn_vt_rows": (C.c_int, [C.c_int]),
    "ldm_gemm_last_config": (C.c_int, [C.POINTER(c_i32), C.POINTER(c_i32), C.POINTER(c_i32)]),
    "ldm_groupnorm_silu": (C.c_int, [C.POINTER(GroupNormDesc), c_vp]),
    "ldm_groupnorm_scratch_bytes": (C.c_size_t, [c_i32, c_i32]),
    "ldm_layernorm": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_vp]),
    "ldm_timestep_sinusoid": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp]),
    "ldm_gemv_bf16": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "ldm_conv3x3_small_cin": (C.c_int, [c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32,
                                        c_i32, c_vp]),
    "ldm_conv3x3_small_cin_act": (C.c_int, [c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32,
                                        c_i32, c_i32, c_vp]),
    "ldm_conv3x3_small_cin_affine": (C.c_int, [c_vp, c_vp, c_vp, c_i32, c_i32, c_f32, c_f32, c_vp, c_vp, c_vp, c_i32, c_i32,
                                               c_i32, c_i32, c_i32, c_vp]),
    "ldm_im2col3x3_s2_pad": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "ldm_softmax_rows": (C.c_int, [c_vp, c_vp, c_i64, c_i32, c_i64, c_i64, c_f32, c_vp]),
    "ldm_resize_bilinear_planar": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "ldm_conv_out": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "ldm_ddim_step": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "ldm_ddim_step_cfg": (C.c_int, [c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "ldm_ddim_step_clip": (C.c_int, [c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_f32, c_i32, c_vp]),
    "ldm_dpmpp_step": (C.c_int, [c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "ldm_unipc_step": (C.c_int, [c_vp, c_vp, c_f32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i64,
                                 c_vp]),
    "ldm_timestep_sinusoid_rows": (C.c_int, [c_vp, c_vp, c_vp, c_i32, c_i32, c_vp]),
    "ldm_gemv_bf16_rows": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_vp]),
    "ldm_ddim_step_rows": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "ldm_dpmpp_step_rows": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "ldm_unipc_step_rows": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i64, c_i64, c_vp]),
    "ldm_upsample_nearest": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "ldm_im2col3x3_s2": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "ldm_logits_to_ids": (C.c_int, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_f32, c_i32, c_vp]),
    "ldm_bilinear_up_nchw": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_vp]),
    "ldm_resize_bilinear_nhwc": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32,
                                           c_i32, c_vp]),
    "ldm_segment_filter": (C.c_int, [c_vp, c_vp, c_vp, c_i32, c_i64, c_i32, c_i32, c_f64, c_i32, c_vp]),
    "ldm_decode_bitmap": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i64, c_i32, c_vp]),
    "ldm_encode_bitmap": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_i64, c_i32, c_f32, c_vp]),
    "ldm_ccl_scratch_bytes": (C.c_size_t, [c_i32, c_i32, c_i32]),
    "ldm_ccl_label4": (C.c_int, [c_vp, c_i32, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "ldm_joint_hist": (C.c_int, [c_vp, c_vp, c_i64, c_vp, c_vp, c_i32, c_vp, c_vp]),
    "ldm_city_pan_scratch_bytes": (C.c_size_t, [c_i32, c_i32, c_i32, c_i32]),
    "ldm_city_pan_maps": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_vp, c_i32, c_i32, c_i32, c_vp]),
    "ldm_joint_hist_batch": (C.c_int, [c_vp, c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_i32, c_vp, c_vp]),
    "ldm_pan_insert": (C.c_int, [c_vp, c_vp, c_i32, c_i32, c_vp, c_i64, c_vp]),
    "ldm_pan_combine": (C.c_int, [c_vp, c_vp, c_i32, c_vp, c_i64, c_vp]),
    "ldm_id_mask": (C.c_int, [c_vp, c_vp, c_i32, c_vp, c_i32, c_i32, c_i64, c_vp]),
    "ldm_depth_mask_pred": (C.c_int, [c_vp, c_i32, c_vp, c_vp, c_i32, c_i32, c_i32, C.c_double, c_i32, c_vp, c_vp, c_i32,
                                      c_vp]),
}

_lib = None


class LdmError(RuntimeError):
    pass


def load():
    """dlopen the library and bind every declared symbol. Raises if the .so has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LdmError(
                f"{LIB_PATH} is missing: build it with `python -m video_latent_diffusion_panoptic_segmentation_b200.build`"
                " (there is no CPU fallback for the sampler hot path)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if lib.ldm_abi_version() != ABI_VERSION:
            raise LdmError(f"{LIB_PATH} has ABI version {lib.ldm_abi_version()}, this binding expects {ABI_VERSION}: "
                           "rebuild it (python -m video_latent_diffusion_panoptic_segmentation_b200.build)")
        _lib = lib
    return _lib


def lib():
    """Library handle for compute calls: additionally requires a B200 (sm_100) as the current CUDA device."""
    l = load()
    rc = l.ldm_check_device()   # the CURRENT device, every time (a process may drive several; the check is two cached queries)
    if rc != 0:
        raise LdmError(f"ldm_check_device failed ({rc}): {l.ldm_last_error().decode()}")
    return l


def check(rc, what=""):
    if rc != 0:
        raise LdmError(f"{what} failed with status {rc}: {load().ldm_last_error().decode()}")


def launch_count():
    return int(load().ldm_launch_count())
