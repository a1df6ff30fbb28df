"""ctypes binding of include/neo360_b200.h (the C ABI of libneo360_b200.so).

The product path has no CPU fallback: importing the renderer without the shared library, or calling it
without a CUDA device, raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libneo360_b200.so")

NEO_PREC_FP32 = 0
NEO_PREC_TC = 1

fp = C.POINTER(C.c_float)


class NeoMLPParams(C.Structure):
    _fields_ = [("in_ch", C.c_int)] + [(n, C.c_void_p) for n in (
        "w0", "b0", "w1", "b1", "w2", "b2", "w3", "b3", "wb", "bb", "wsig", "bsig", "wv0", "bv0", "wv1", "bv1",
        "wrgb", "brgb")]


class NeoSceneDesc(C.Structure):
    _fields_ = [("nv", C.c_int), ("plane_h", C.c_int), ("plane_w", C.c_int), ("world_ch", C.c_int),
                ("lat_h", C.c_int), ("lat_w", C.c_int), ("local_ch", C.c_int), ("img_w", C.c_int), ("img_h", C.c_int),
                ("planes_xz", C.c_void_p), ("planes_xy", C.c_void_p), ("planes_yz", C.c_void_p),
                ("latent", C.c_void_p), ("src_poses", C.c_void_p), ("src_focal", C.c_void_p), ("src_c", C.c_void_p)]


class NeoRays(C.Structure):
    _fields_ = [("n_rays", C.c_int), ("chunk", C.c_int), ("rays_o", C.c_void_p), ("rays_d", C.c_void_p),
                ("viewdirs", C.c_void_p), ("ray_order", C.c_void_p)]


class NeoCfg(C.Structure):
    _fields_ = [("n_coarse", C.c_int), ("n_fine", C.c_int), ("white_bkgd", C.c_int), ("out_depth", C.c_int),
                ("precision", C.c_int), ("u_fg0", C.c_void_p), ("u_bg0", C.c_void_p), ("u_fg1", C.c_void_p),
                ("u_bg1", C.c_void_p)]


OUT_FIELDS = ("comp_rgb", "fg_rgb", "bg_rgb", "fg_acc", "bg_lambda", "depth", "bg_acc", "fg_w", "bg_w", "fg_sdist",
              "bg_sdist", "fg_t", "bg_s", "fg_sigma", "bg_sigma", "fg_rgb_s", "bg_rgb_s")


class NeoOut(C.Structure):
    _fields_ = [(n, C.c_void_p * 2) for n in OUT_FIELDS]


class NeoVanillaMLPParams(C.Structure):
    _fields_ = [("w", C.c_void_p * 8), ("b", C.c_void_p * 8)] + [(n, C.c_void_p) for n in ("wb", "bb", "wsig", "bsig", "wv0", "bv0", "wrgb", "brgb")]


class NeoVanillaCfg(C.Structure):
    _fields_ = [("n_coarse", C.c_int), ("n_fine", C.c_int), ("white_bkgd", C.c_int), ("near_plane", C.c_float), ("far_plane", C.c_float),
                ("u0", C.c_void_p), ("u1", C.c_void_p), ("precision", C.c_int)]


VANILLA_OUT_FIELDS = ("comp_rgb", "acc", "depth", "t", "sigma", "rgb_s", "weights")


class NeoVanillaOut(C.Structure):
    _fields_ = [(n, C.c_void_p * 2) for n in VANILLA_OUT_FIELDS]


class NeoMipMLPParams(C.Structure):
    _fields_ = [("depth", C.c_int), ("width", C.c_int), ("basis", C.c_void_p), ("w", C.c_void_p * 8), ("b", C.c_void_p * 8)] + \
               [(n, C.c_void_p) for n in ("wsig", "bsig", "wb", "bb", "wv0", "bv0", "wrgb", "brgb")]


class NeoMipCfg(C.Structure):
    _fields_ = [("n_prop", C.c_int), ("n_nerf", C.c_int), ("near_plane", C.c_float), ("far_plane", C.c_float), ("train_frac", C.c_float),
                ("jitter", C.c_void_p * 3), ("precision", C.c_int)]


MIP_OUT_FIELDS = ("rgb", "density", "rgb_s", "sdist", "weights")


class NeoMipOut(C.Structure):
    _fields_ = [(n, C.c_void_p * 3) for n in MIP_OUT_FIELDS]


class NeoGridEncoderParams(C.Structure):
    _fields_ = [("fc_w", C.c_void_p * 3), ("fc_b", C.c_void_p * 3)] + \
               [(f"agg_{pl}_{n}", C.c_void_p) for pl in ("xz", "yz", "xy") for n in ("w0", "b0", "w1", "b1")]


# every symbol include/neo360_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "neo_scene_create": (C.c_int, [C.POINTER(NeoSceneDesc), C.POINTER(NeoMLPParams), C.c_int, C.POINTER(C.c_void_p), C.c_void_p]),
    "neo_scene_free": (None, [C.c_void_p]),
    "neo_scene_bytes": (C.c_size_t, [C.c_void_p]),
    "neo_render_workspace_bytes": (C.c_size_t, [C.c_int, C.POINTER(NeoCfg)]),
    "neo_render_fwd": (C.c_int, [C.c_void_p, C.POINTER(NeoRays), C.POINTER(NeoCfg), C.POINTER(NeoOut), C.c_void_p, C.c_size_t, C.c_void_p]),
    "neo_check_async": (C.c_int, [C.c_void_p, C.c_void_p]),
    "neo_sample_rays": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_release_cached": (None, []),
    "neo_index_maps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_index_maps_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "neo_get_rays": (C.c_int, [C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_intersect_sphere": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_sample_along_rays": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_sample_pdf": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_volumetric_rendering": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_index_grid": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "neo_index_local": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "neo_clipped_sq_err": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "neo_volumetric_rendering_bwd": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 4 + [C.c_void_p] * 8),
    "neo_index_grid_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_index_local_bwd": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_field_eval": (C.c_int, [C.c_void_p, C.POINTER(NeoRays), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_vanilla_create": (C.c_int, [C.POINTER(NeoVanillaMLPParams), C.POINTER(C.c_void_p), C.c_void_p]),
    "neo_vanilla_free": (None, [C.c_void_p]),
    "neo_vanilla_workspace_bytes": (C.c_size_t, [C.c_int, C.POINTER(NeoVanillaCfg)]),
    "neo_vanilla_render_fwd": (C.c_int, [C.c_void_p, C.POINTER(NeoRays), C.POINTER(NeoVanillaCfg), C.POINTER(NeoVanillaOut), C.c_void_p, C.c_size_t, C.c_void_p]),
    "neo_mip_workspace_bytes": (C.c_size_t, [C.c_int, C.POINTER(NeoMipCfg), C.c_int]),
    "neo_mip_render_fwd": (C.c_int, [C.POINTER(NeoMipMLPParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(NeoMipCfg),
                                     C.POINTER(NeoMipOut), C.c_void_p, C.c_size_t, C.c_void_p]),
    "neo_grid_encoder_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "neo_grid_encoder_dense": (C.c_int, [C.POINTER(NeoGridEncoderParams), C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "neo_profile": (C.c_int, [C.c_int]),
    "neo_profile_read": (C.c_int, [C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_ulonglong), C.POINTER(C.c_double)]),
    "neo_tc_selftest": (C.c_int, [C.c_void_p] * 8),
    "neo_tc_selftest_transpose": (C.c_int, [C.c_void_p] * 4),
    "neo_tc_dense": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "neo_tc_enc_column": (C.c_int, [C.c_int, C.c_int]),
    "neo_tc_debug": (C.c_int, [C.c_void_p]),
    "neo_tc_selftest_window": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "neo_tc_trap_info": (C.c_char_p, []),
    "neo_last_error": (C.c_char_p, []),
    "neo_version": (C.c_char_p, []),
}

_lib = None


def load(path=None):
    """dlopen the library at `path` (default: the in-tree one) and type its entry points; the first call decides which
    library the process uses.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("NEO360_B200_LIB") or path or LIB_PATH      # override: A/B runs of experimental kernel builds (tools/)
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -m neo360_b200.build` (or __graft_entry__.build()); "
                           "there is no CPU fallback")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError(f"neo360_b200 error {rc}: {load().neo_last_error().decode()}{load().neo_tc_trap_info().decode()}")


def ptr(t):
    """device pointer of a contiguous fp32 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    import torch
    if not (t.is_cuda and t.is_contiguous() and t.dtype in (torch.float32, torch.int32, torch.uint8)):
        raise ValueError("neo360_b200 takes contiguous fp32 CUDA tensors")
    return t.data_ptr()
