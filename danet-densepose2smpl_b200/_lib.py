"""ctypes binding of libdanet_b200.so (the C ABI in include/danet_b200.h).

There is no CPU fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdanet_b200.so")

c_int, c_i64, c_f, c_p = ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p


class SmplDesc(ctypes.Structure):
    _fields_ = [("num_verts", c_int), ("num_joints", c_int), ("num_betas", c_int),
                ("v_template", c_p), ("shapedirs", c_p), ("posedirs", c_p), ("J_regressor", c_p),
                ("lbs_weights", c_p), ("parents", c_p),
                ("num_selected", c_int), ("selected_verts", c_p),
                ("num_extra", c_int), ("J_regressor_extra", c_p),
                ("num_h36m", c_int), ("J_regressor_h36m", c_p),
                ("num_out_joints", c_int), ("joint_map", c_p)]


class RasterDesc(ctypes.Structure):
    _fields_ = [("num_smpl_verts", c_int), ("num_mesh_verts", c_int), ("vert_mapping", c_p),
                ("num_faces", c_int), ("faces", c_p), ("textures", c_p),
                ("orig_size", c_int), ("out_size", c_int), ("focal_length", c_f),
                ("near_plane", c_f), ("far_plane", c_f), ("tex_mode", c_int)]


class ConvDesc(ctypes.Structure):
    _fields_ = [("N", c_int), ("H", c_int), ("W", c_int), ("Cin", c_int), ("Cout", c_int),
                ("ksize", c_int), ("stride", c_int), ("pad", c_int), ("wsets", c_int), ("relu", c_int), ("flags", c_int)]


class Act(ctypes.Structure):
    """danet_act: fp32 view and/or split-fp16 planes of one NHWC activation tensor."""
    _fields_ = [("f32", c_p), ("hi", c_p), ("lo", c_p)]


class ConvProblem(ctypes.Structure):
    _fields_ = [("d", ConvDesc), ("x", Act), ("res", Act), ("y", Act), ("w_packed", c_p), ("bias", c_p)]


class GcnParams(ctypes.Structure):
    _fields_ = [("adj", c_p), ("W", c_p * 5), ("b", c_p * 5), ("bn_scale", c_p * 5),
                ("bn_shift", c_p * 5), ("dim_in", c_int * 5), ("dim_out", c_int * 5),
                ("head_w", c_p), ("head_b", c_p), ("mean_pose", c_p)]


# name -> (restype, argtypes); every symbol include/danet_b200.h declares
SIGNATURES = {
    "danet_last_error": (ctypes.c_char_p, []),
    "danet_version": (c_int, []),
    "danet_device_info": (c_int, [c_p, c_p, c_p]),
    "danet_smpl_create": (c_int, [ctypes.POINTER(SmplDesc), ctypes.POINTER(c_p)]),
    "danet_smpl_destroy": (c_int, [c_p]),
    "danet_smpl_workspace_bytes": (c_i64, [c_p, c_int]),
    "danet_smpl_forward": (c_int, [c_p, c_int, c_p, c_p, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p]),
    "danet_smpl_backward_workspace_bytes": (c_i64, [c_p, c_int]),
    "danet_smpl_backward": (c_int, [c_p, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_rot6d_to_rotmat": (c_int, [c_int, c_p, c_p, c_p]),
    "danet_batch_rodrigues": (c_int, [c_int, c_p, c_p, c_int, c_p]),
    "danet_perspective_projection": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_mpjpe_h36m": (c_int, [c_int, c_p, c_p, c_p, c_p]),
    "danet_body_uv_losses_workspace_bytes": (c_i64, [c_int, c_int]),
    "danet_body_uv_losses": (c_int, [c_int, c_int, c_int, c_int, c_i64, c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                                     c_p, c_f, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_dp_uvia_losses_workspace_bytes": (c_i64, [c_int, c_int, c_int, c_int]),
    "danet_dp_uvia_losses": (c_int, [c_int, c_int, c_int, c_int, c_int] + [c_p] * 12 + [c_int, c_f, c_f, c_f]
                             + [c_p] * 7),
    "danet_stn_kps_losses_workspace_bytes": (c_i64, [c_int, c_int]),
    "danet_stn_kps_losses": (c_int, [c_int, c_int, c_int, c_p, c_p, c_f, c_p, c_p, c_p, c_p, c_p]),
    "danet_raster_create": (c_int, [ctypes.POINTER(RasterDesc), ctypes.POINTER(c_p)]),
    "danet_raster_destroy": (c_int, [c_p]),
    "danet_raster_workspace_bytes": (c_i64, [c_p, c_int]),
    "danet_raster_iuv": (c_int, [c_p, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_iuv_img2map": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_conv2d": (c_int, [ctypes.POINTER(ConvDesc), c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_conv_tc_packed_bytes": (c_i64, [ctypes.POINTER(ConvDesc)]),
    "danet_conv_tc_pack": (c_int, [ctypes.POINTER(ConvDesc), c_p, c_p, c_p]),
    "danet_conv_tc_supported": (c_int, [ctypes.POINTER(ConvDesc)]),
    "danet_conv_tc_group": (c_int, [c_int, ctypes.POINTER(ConvProblem), c_p]),
    "danet_conv_tc_config": (c_int, [c_int, ctypes.POINTER(ConvDesc), c_p, c_p]),
    "danet_conv_tc_set_profile_buffer": (c_int, [c_p]),
    "danet_act_split": (c_int, [c_i64, c_p, c_p, c_p, c_p]),
    "danet_act_merge": (c_int, [c_i64, c_p, c_p, c_p, c_p]),
    "danet_nchw_to_nhwc": (c_int, [c_int, c_int, c_int, c_int, c_p, ctypes.POINTER(Act), c_p]),
    "danet_fuse_sum": (c_int, [c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(Act), c_p, c_int, ctypes.POINTER(Act), c_p]),
    "danet_maxpool3x3s2": (c_int, [c_int, c_int, c_int, c_int, ctypes.POINTER(Act), ctypes.POINTER(Act), c_p]),
    "danet_global_avgpool": (c_int, [c_int, c_int, c_int, ctypes.POINTER(Act), c_p, c_p]),
    "danet_linear": (c_int, [c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_iuv_clean_global": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_p, ctypes.POINTER(Act), c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_iuvmap_clean_nchw": (c_int, [c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "danet_iuv_clean_parts": (c_int, [c_int, c_int, c_int, c_int, c_p, ctypes.POINTER(Act), c_p, c_p]),
    "danet_stn_params": (c_int, [c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_f, c_int, c_p, c_p, c_p]),
    "danet_stn_sample": (c_int, [c_int, c_int, c_int, ctypes.POINTER(Act), c_p, c_int, ctypes.POINTER(Act), c_p]),
    "danet_gcn_pose_head": (c_int, [c_int, ctypes.POINTER(GcnParams), c_p, c_p, c_p, c_p]),
    "danet_net_load": (c_int, [c_p, ctypes.c_uint64, ctypes.POINTER(c_p)]),
    "danet_net_load_file": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_p)]),
    "danet_net_destroy": (c_int, [c_p]),
    "danet_net_info": (c_int, [c_p, c_p, c_p, c_p, c_p]),
    "danet_net_output_name": (ctypes.c_char_p, [c_p, c_int]),
    "danet_net_output": (c_int, [c_p, ctypes.c_char_p, ctypes.POINTER(c_p), ctypes.POINTER(ctypes.c_uint64), c_p, c_p]),
    "danet_net_infer": (c_int, [c_p, c_p, c_int, c_p]),
    "danet_net_infer_host": (c_int, [c_p, c_p, c_int]),
    "danet_net_read_output": (c_int, [c_p, ctypes.c_char_p, c_p, ctypes.c_uint64]),
}

_lib = None


def load():
    """Load libdanet_b200.so (once) and bind every signature.  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "danet_b200: %s not found -- build it with `python __graft_entry__.py` "
                "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = load().danet_last_error()
        raise RuntimeError("danet_b200 %s failed (rc=%d): %s" % (what, rc, msg.decode() if msg else "?"))


def stream_ptr(device=None):
    """Current torch stream of `device` (default: the current device).  Callers that own a device pass it
    and launch under `torch.cuda.device(device)` so that kernels, pointers and stream agree."""
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return ctypes.c_void_p(0)
    return ctypes.c_void_p(t.data_ptr())


def require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError("danet_b200: %s must be a CUDA tensor (there is no CPU path)" % name)
