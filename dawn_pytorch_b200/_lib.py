"""ctypes binding of include/dawn_unet.h.  The product path has no fallback: if the CUDA library is
missing or fails to load, importing this module raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdawn_unet.so")


class DawnUnetCfg(ctypes.Structure):
    _fields_ = [("dim", ctypes.c_int), ("n_levels", ctypes.c_int), ("dim_mults", ctypes.c_int * 8),
                ("channels", ctypes.c_int), ("cond_aud", ctypes.c_int), ("cond_pose", ctypes.c_int),
                ("cond_eye", ctypes.c_int), ("out_grid_dim", ctypes.c_int), ("out_conf_dim", ctypes.c_int),
                ("attn_heads", ctypes.c_int), ("attn_dim_head", ctypes.c_int), ("resnet_groups", ctypes.c_int),
                ("init_kernel_size", ctypes.c_int), ("win_width", ctypes.c_int)]


class DawnLfgCfg(ctypes.Structure):
    """include/dawn_lfg.h: dawn_lfg_cfg"""
    _fields_ = [("num_channels", ctypes.c_int), ("block_expansion", ctypes.c_int), ("max_features", ctypes.c_int),
                ("num_down_blocks", ctypes.c_int), ("num_bottleneck_blocks", ctypes.c_int), ("skips", ctypes.c_int)]


class DawnError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python dawn_pytorch_b200/build.py` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for the DAWN denoising UNet.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i64p, fp, cp = ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.c_void_p, ctypes.c_char_p
    lib.dawn_unet_create.argtypes = [ctypes.POINTER(DawnUnetCfg), ctypes.POINTER(vp)]
    lib.dawn_unet_destroy.argtypes = [vp]
    lib.dawn_unet_destroy.restype = None
    lib.dawn_unet_set_param.argtypes = [vp, cp, fp, i64p, ctypes.c_int]
    lib.dawn_unet_commit_params.argtypes = [vp]
    lib.dawn_unet_set_num_frames.argtypes = [vp, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.dawn_unet_set_clip_invariants.argtypes = [vp, fp, fp, vp]
    lib.dawn_unet_forward.argtypes = [vp, fp, vp, fp, fp, vp]
    lib.dawn_unet_forward_x3.argtypes = [vp, fp, vp, fp, vp]
    lib.dawn_unet_forward_host.argtypes = [vp, fp, fp, fp, ctypes.c_int64, fp]
    lib.dawn_unet_set_tap.argtypes = [vp, cp, fp]
    lib.dawn_unet_tap_shape.argtypes = [vp, cp, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int),
                                        ctypes.POINTER(ctypes.c_int)]
    dp = ctypes.POINTER(ctypes.c_double)
    lib.dawn_unet_profile_enable.argtypes = [vp, ctypes.c_int]
    lib.dawn_unet_profile_read.argtypes = [vp, dp, dp, dp, i64p]
    lib.dawn_unet_last_launch_count.argtypes = [vp]
    lib.dawn_unet_last_launch_count.restype = ctypes.c_int64
    lib.dawn_unet_workspace_bytes.argtypes = [vp]
    lib.dawn_unet_workspace_bytes.restype = ctypes.c_int64
    lib.dawn_selftest_tc_gemm.argtypes = [ctypes.c_int] * 7 + [ctypes.POINTER(ctypes.c_float)] * 2
    lib.dawn_selftest_attention.argtypes = [ctypes.c_int] * 3 + [ctypes.POINTER(ctypes.c_float)] * 2
    lib.dawn_temporal_tc_plan.argtypes = [ctypes.c_int] * 4 + [ctypes.POINTER(ctypes.c_int)]
    lib.dawn_selftest_temporal_tc.argtypes = [ctypes.c_int] * 5 + [ctypes.POINTER(ctypes.c_float)] * 2 + [ctypes.POINTER(ctypes.c_uint64), ctypes.POINTER(ctypes.c_float)]
    lib.dawn_nccl_unique_id.argtypes = [ctypes.c_char_p]
    lib.dawn_unet_init_shard.argtypes = [vp, ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]
    lib.dawn_unet_shard_ipc_export.argtypes = [vp, ctypes.c_char_p]
    lib.dawn_unet_shard_ipc_import.argtypes = [vp, ctypes.c_char_p]
    lib.dawn_ddim_step.argtypes = [fp, fp, fp, ctypes.c_int64] + [ctypes.c_float] * 6 + [vp, vp]
    lib.dawn_unet_ddim_step.argtypes = [vp, fp, fp, fp, ctypes.c_int64] + [ctypes.c_float] * 6 + [vp, vp]
    lib.dawn_unet_sampler_capture.argtypes = [vp, fp, fp, fp, vp, ctypes.POINTER(ctypes.c_float), ctypes.c_int, ctypes.c_float, vp]
    lib.dawn_unet_sampler_launch.argtypes = [vp, vp]
    lib.dawn_unet_ddpm_step.argtypes = [vp, fp, fp, fp, ctypes.c_int64, fp, ctypes.c_float, vp, vp]
    lib.dawn_unet_ddpm_capture.argtypes = [vp, fp, fp, fp, vp, vp, vp, ctypes.c_int, ctypes.c_float, vp]
    ip = ctypes.POINTER(ctypes.c_int)
    lib.dawn_lfg_create.argtypes = [ctypes.POINTER(DawnLfgCfg), ctypes.POINTER(vp)]
    lib.dawn_lfg_destroy.argtypes = [vp]
    lib.dawn_lfg_destroy.restype = None
    lib.dawn_lfg_set_param.argtypes = [vp, cp, fp, i64p, ctypes.c_int]
    lib.dawn_lfg_commit_params.argtypes = [vp]
    lib.dawn_lfg_set_geometry.argtypes = [vp] + [ctypes.c_int] * 5
    lib.dawn_lfg_set_source.argtypes = [vp, fp, vp]
    lib.dawn_lfg_get_fea.argtypes = [vp, fp, vp]
    lib.dawn_lfg_decode.argtypes = [vp, fp, fp, fp, fp, vp]
    lib.dawn_lfg_decode_sample.argtypes = [vp, fp, fp, fp, vp]
    lib.dawn_lfg_read_tap.argtypes = [vp, cp, fp, ip, ip, ip, vp]
    lib.dawn_conv3x3_s2_relu.argtypes = [fp, ctypes.c_int, ctypes.c_int, ctypes.c_int, fp, fp, ctypes.c_int, fp, vp]
    lib.dawn_lfg_last_launch_count.argtypes = [vp]
    lib.dawn_lfg_last_launch_count.restype = ctypes.c_int64
    lib.dawn_lfg_workspace_bytes.argtypes = [vp]
    lib.dawn_lfg_workspace_bytes.restype = ctypes.c_int64
    lib.dawn_last_error.restype = cp
    lib.dawn_build_info.restype = cp
    return lib


lib = _load()

EXPORTS = ["dawn_unet_create", "dawn_unet_destroy", "dawn_unet_set_param", "dawn_unet_commit_params",
           "dawn_unet_set_num_frames", "dawn_nccl_unique_id", "dawn_unet_init_shard", "dawn_unet_shard_ipc_export", "dawn_unet_shard_ipc_import", "dawn_unet_set_clip_invariants", "dawn_unet_forward",
           "dawn_unet_forward_x3", "dawn_unet_forward_host", "dawn_unet_set_tap", "dawn_unet_tap_shape",
           "dawn_unet_profile_enable", "dawn_unet_profile_read", "dawn_unet_last_launch_count", "dawn_unet_workspace_bytes", "dawn_ddim_step", "dawn_unet_ddim_step", "dawn_unet_sampler_capture", "dawn_unet_sampler_launch",
           "dawn_unet_ddpm_step", "dawn_unet_ddpm_capture",
           "dawn_selftest_tc_gemm", "dawn_selftest_attention", "dawn_selftest_temporal_tc", "dawn_temporal_tc_plan", "dawn_last_error", "dawn_build_info"]


LFG_EXPORTS = ["dawn_lfg_create", "dawn_lfg_destroy", "dawn_lfg_set_param", "dawn_lfg_commit_params", "dawn_lfg_set_geometry",
               "dawn_lfg_set_source", "dawn_lfg_get_fea", "dawn_lfg_decode", "dawn_lfg_decode_sample", "dawn_lfg_read_tap",
               "dawn_lfg_last_launch_count", "dawn_lfg_workspace_bytes"]
MISC_EXPORTS = ["dawn_conv3x3_s2_relu"]

PROF_CATS = ["conv3x3", "conv_other", "qkv_proj", "out_proj", "ca_gate", "gn_hcond", "attn_core", "sla_context",
             "gn_apply", "rowstats", "ca_rstd", "misc", "prep", "temporal_fused_l0", "conv3x3_l0", "comm_allreduce", "comm_halo"]
PROF_NCAT = 20


def check(rc, what):
    if rc != 0:
        raise DawnError(f"{what} failed (rc={rc}): {lib.dawn_last_error().decode()}")
