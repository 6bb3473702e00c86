"""ctypes binding of libmi3d.so (C ABI declared in include/mi3d.h).

The product path has NO fallback: if the shared library is missing, or a call returns non-zero, we raise.
"""
import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MI3D_LIB_PATH") or os.path.join(_HERE, "libmi3d.so")      # override: A/B builds under tools/
_lib = None


class Mi3dError(RuntimeError):
    pass


class HashGrid(C.Structure):
    _fields_ = [("n_levels", C.c_uint32), ("n_entries", C.c_uint32), ("offsets", C.c_uint32 * 16),
                ("sizes", C.c_uint32 * 16), ("ress", C.c_uint32 * 16), ("scales", C.c_float * 16)]


class RayGen(C.Structure):
    _fields_ = [("cams", C.c_void_p), ("n_views", C.c_uint32), ("H", C.c_uint32), ("W", C.c_uint32), ("rays_per_view", C.c_uint32),
                ("pixel_stride", C.c_uint32), ("pixel_phase", C.c_uint32)]


class Mlp(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("w1", "b1", "w2", "b2", "w3", "b3")]


class Epilogue(C.Structure):
    _fields_ = [("bg_color", C.c_void_p), ("bg_scalar", C.c_float), ("max_depth", C.c_float), ("depth_scale", C.c_void_p),
                ("rays_per_view", C.c_uint32)]


class FieldCfg(C.Structure):
    _fields_ = [("bound", C.c_float), ("blob_density", C.c_float), ("blob_radius", C.c_float), ("n_evals", C.c_int),
                ("shading", C.c_int), ("ambient_ratio", C.c_float), ("light_d", C.c_void_p), ("impl", C.c_int), ("scatter_agg_scale", C.c_float)]


class FieldIO(C.Structure):
    _fields_ = [("xyzs", C.c_void_p), ("dirs", C.c_void_p), ("counter", C.c_void_p), ("m_fixed", C.c_uint32),
                ("align", C.c_uint32), ("cap", C.c_uint32), ("smooth_noise", C.c_void_p), ("seed", C.c_uint64),
                ("enc_cache", C.c_void_p), ("enc_cache_tiles", C.c_uint32), ("enc_cache_valid", C.c_uint32),
                ("segs", C.c_void_p), ("n_views", C.c_uint32), ("noise_mode", C.c_uint32)]


MAX_VIEWS = 8


class ViewSegs(C.Structure):
    _fields_ = [("n_views", C.c_uint32), ("bounds", C.c_uint32 * (2 * MAX_VIEWS + 1)), ("mpad", C.c_uint32 * MAX_VIEWS)]


class AdanCfg(C.Structure):
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("beta3", C.c_double), ("eps", C.c_double),
                ("weight_decay", C.c_double), ("max_grad_norm", C.c_float), ("clip_grad_norm", C.c_float), ("no_prox", C.c_int),
                ("step", C.c_int), ("reset_prev", C.c_int)]


class RenderArgs(C.Structure):
    _fields_ = [("rays_o", C.c_void_p), ("rays_d", C.c_void_p), ("depth_scale", C.c_void_p), ("raygen", C.POINTER(RayGen)), ("N", C.c_uint32),
                ("n_views", C.c_uint32), ("density_bitfield", C.c_void_p), ("C", C.c_uint32), ("H", C.c_uint32), ("bound", C.c_float),
                ("dt_gamma", C.c_float), ("max_steps", C.c_uint32), ("min_near", C.c_float), ("aabb", C.c_void_p), ("noises", C.c_void_p),
                ("seed", C.c_uint64), ("T_thresh", C.c_float), ("bg_color", C.c_void_p), ("bg_scalar", C.c_float), ("max_depth", C.c_float),
                ("smooth_noise", C.c_void_p), ("noise_mode", C.c_uint32), ("all_counts", C.c_void_p), ("n_ranks", C.c_uint32),
                ("pad_view_mask", C.c_uint32)]


class RenderEvalArgs(C.Structure):
    _fields_ = [("rays_o", C.c_void_p), ("rays_d", C.c_void_p), ("depth_scale", C.c_void_p), ("N", C.c_uint32), ("density_bitfield", C.c_void_p),
                ("C", C.c_uint32), ("H", C.c_uint32), ("bound", C.c_float), ("dt_gamma", C.c_float), ("max_steps", C.c_uint32), ("min_near", C.c_float),
                ("aabb", C.c_void_p), ("T_thresh", C.c_float), ("perturb", C.c_int), ("seed", C.c_uint64), ("bg_color", C.c_void_p),
                ("bg_scalar", C.c_float), ("max_depth", C.c_float)]


class RenderWs(C.Structure):
    _fields_ = [("N", C.c_uint32), ("cap", C.c_uint32), ("n_views", C.c_uint32)] + \
               [(n, C.c_void_p) for n in ("xyzs", "dirs", "deltas", "sigmas", "rgbs", "tape", "g_sigmas", "g_rgbs", "rays", "counter", "nears",
                                          "fars", "ws_raw", "depth_raw", "image_raw", "depth_scale", "scan_ws", "loss_partials", "view_counts",
                                          "segs", "enc_cache")] + [("enc_cache_tiles", C.c_uint32), ("bytes", C.c_size_t)]


RENDER_PHASE_MARCH, RENDER_PHASE_SHADE, RENDER_PHASE_ALL = 1, 2, 3

SHADING = {"albedo": 0, "lambertian": 1, "textureless": 2, "normal": 3}
FIELD_IMPL = {"tcgen05": 0, "ffma": 1, "tcgen05_fused_scatter": 2, "tcgen05_split_scatter": 3, "tcgen05_single_e": 4}

# every symbol include/mi3d.h declares (tests/test_abi.py checks the .so exports exactly these)
SYMBOLS = [
    "mi3d_near_far_from_aabb", "mi3d_morton3D", "mi3d_morton3D_invert", "mi3d_packbits",
    "mi3d_march_rays_train_workspace_bytes", "mi3d_march_rays_train", "mi3d_march_rays_train_cam", "mi3d_get_rays",
    "mi3d_composite_rays_train_forward", "mi3d_composite_rays_train_backward",
    "mi3d_march_rays", "mi3d_composite_rays",
    "mi3d_hashgrid_make", "mi3d_hashgrid_forward", "mi3d_hashgrid_backward",
    "mi3d_field_grid_ctas", "mi3d_field_forward", "mi3d_field_backward", "mi3d_field_backward_workspace_bytes", "mi3d_field_enc_cache_bytes",
    "mi3d_render_workspace_bytes", "mi3d_render_workspace_carve", "mi3d_render_forward", "mi3d_render_backward",
    "mi3d_render_eval_workspace_bytes", "mi3d_render_eval",
    "mi3d_density_grid_workspace_bytes", "mi3d_density_grid_update", "mi3d_version",
    "mi3d_sumsq_workspace_bytes", "mi3d_sumsq", "mi3d_adan_step",
    "mi3d_gemm_f16", "mi3d_gemm_f16_splitk", "mi3d_flash_attn_f16", "mi3d_conv3x3_f16", "mi3d_tf32_tile_test", "mi3d_gemm_f16_bt",
    "mi3d_sd_workspace_bytes", "mi3d_sd_create", "mi3d_sd_destroy", "mi3d_sd_num_params", "mi3d_sd_param_name", "mi3d_sd_param_numel",
    "mi3d_sd_param_shape", "mi3d_sd_load_param", "mi3d_sd_encode", "mi3d_sd_encode_backward", "mi3d_sd_unet_sds", "mi3d_sd_debug_tensor", "mi3d_sd_profile",
    "mi3d_sd_profile_dump", "mi3d_sd_set_graph_replay", "mi3d_sd_graph_replays", "mi3d_sd_ddim_step", "mi3d_sd_decode",
    "mi3d_point_render_workspace_bytes", "mi3d_point_render_forward", "mi3d_point_render_backward",
]


def build(verbose=False):
    """Compile libmi3d.so in-tree with nvcc for sm_100a (no GPU needed)."""
    out = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc")], capture_output=True, text=True)
    if out.returncode != 0:
        raise Mi3dError("building libmi3d.so failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise Mi3dError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU / PyTorch fallback for the hot path)")
        _lib = C.CDLL(LIB_PATH)
        _lib.mi3d_version.restype = C.c_char_p
        _lib.mi3d_march_rays_train_workspace_bytes.restype = C.c_size_t
        _lib.mi3d_density_grid_workspace_bytes.restype = C.c_size_t
        _lib.mi3d_field_backward_workspace_bytes.restype = C.c_size_t
        _lib.mi3d_field_enc_cache_bytes.restype = C.c_size_t
        _lib.mi3d_render_workspace_bytes.restype = C.c_size_t
        _lib.mi3d_sumsq_workspace_bytes.restype = C.c_size_t
        _lib.mi3d_render_eval_workspace_bytes.restype = C.c_size_t
        _lib.mi3d_point_render_workspace_bytes.restype = C.c_size_t
        for name in ("mi3d_sd_workspace_bytes", "mi3d_sd_weight_bytes"):
            if hasattr(_lib, name):
                getattr(_lib, name).restype = C.c_size_t
        if hasattr(_lib, "mi3d_sd_create"):
            _lib.mi3d_sd_create.restype = C.c_void_p
    return _lib


def check(code, what):
    if code != 0:
        if code == 1000001:
            raise Mi3dError(f"{what}: invalid argument (MI3D_ERR_ARG)")
        raise Mi3dError(f"{what}: CUDA error {code}")


def ptr(t):
    """device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise Mi3dError("mi3d kernels need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise Mi3dError("mi3d kernels need contiguous tensors")
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def f32c(t):
    return t.contiguous().float() if (t.dtype != torch.float32 or not t.is_contiguous()) else t


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise Mi3dError("mi3d operators run on sm_100a only; got a CPU tensor and there is no CPU fallback")
