"""ctypes binding of libb200flow.so (the C-ABI declared in include/b200flow.h).

There is no fallback: if the shared library is missing or does not export the ABI this package was written
against, importing rpeflow_b200 fails loudly.  Build it with ``python __graft_entry__.py`` or
``make -C rpeflow_b200/csrc``.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200FLOW_LIB") or os.path.join(_HERE, "libb200flow.so")     # the override is for kernel A/B builds
ABI_VERSION = 8

c_i, c_i64, c_p = ctypes.c_int, ctypes.c_int64, ctypes.c_void_p


class Corr3dWeights(ctypes.Structure):
    """struct b200_corr3d_weights (include/b200flow.h)."""
    NAMES = ("W1", "b1", "W2", "b2",
             "n1_Wa", "n1_ba", "n1_Wb", "n1_bb", "n1_Wc", "n1_bc",
             "n2_Wa", "n2_ba", "n2_Wb", "n2_bb", "n2_Wc", "n2_bc")
    _fields_ = [(n, c_p) for n in NAMES]


class Corr3dGrads(ctypes.Structure):
    """struct b200_corr3d_grads (include/b200flow.h): the 4 input gradients, then the 16 parameter gradients."""
    NAMES = ("xyz1", "feat1", "xyz2", "feat2") + Corr3dWeights.NAMES
    _fields_ = [(n, c_p) for n in NAMES]


class PointConvWeights(ctypes.Structure):
    """struct b200_pointconv_weights (include/b200flow.h)."""
    NAMES = ("Wa", "ba", "Wb", "bb", "L", "bias")
    _fields_ = [(n, c_p) for n in NAMES]


class PointConvGrads(ctypes.Structure):
    """struct b200_pointconv_grads (include/b200flow.h): the 3 input gradients, then the 6 parameter gradients."""
    NAMES = ("xyz", "feat", "sampled_xyz") + PointConvWeights.NAMES
    _fields_ = [(n, c_p) for n in NAMES]


# name -> (restype, argtypes); one entry per symbol declared in include/b200flow.h
SIGNATURES = {
    "b200_abi_version": (c_i, []),
    "b200_build_info": (ctypes.c_char_p, []),
    "b200_last_error": (ctypes.c_char_p, []),
    "b200_corr2d_fwd": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_corr2d_fwd_nchw": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_corr2d_fwd_nchw_leaky": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, ctypes.c_float, c_p]),
    "b200_backwarp2d": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p]),
    "b200_convex_upsample": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p]),
    "b200_backwarp2d_bwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p]),
    "b200_convex_upsample_bwd_scratch_floats": (c_i64, [c_i, c_i, c_i, c_i]),
    "b200_convex_upsample_bwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p]),
    "b200_corr2d_bwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_corr2d_bwd_nchw": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_fps": (c_i, [c_p, c_p, c_i, c_i, c_i, c_p]),
    "b200_fps_scratch_bytes": (c_i64, [c_i, c_i]),
    "b200_fps_large": (c_i, [c_p, c_p, c_p, c_i64, c_i, c_i, c_i, c_p]),
    "b200_knn": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_knn_scratch_bytes": (c_i64, [c_i, c_i, c_i, c_i, c_i]),
    "b200_knn_grid": (c_i, [c_p, c_p, c_p, c_p, c_i64, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_knn_grid_cf": (c_i, [c_p, c_p, c_p, c_p, c_i64, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_gather_cf": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i64, c_p, c_p]),
    "b200_gather_cl": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i64, c_p, c_p]),
    "b200_grid_sample_pts": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_grid_sample_pts_bwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_gather_cf_bwd": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i64, c_p]),
    "b200_gather_cl_bwd": (c_i, [c_p, c_p, c_p, c_i, c_i, c_i, c_i64, c_p]),
    "b200_project_nn_corr": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_project_nn_corr_scratch_floats": (c_i64, [c_i, c_i, c_i, c_i]),
    "b200_project_nn_corr_sampled": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_pointconv_scratch_floats": (c_i64, [c_i, c_i, c_i, c_i]),
    "b200_pointconv_fwd": (c_i, [c_p, c_p, c_p, c_p, ctypes.POINTER(PointConvWeights), c_p, c_p,
                                 c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_pointconv_fwd_linear": (c_i, [c_p, c_p, c_p, c_p, ctypes.POINTER(PointConvWeights), c_p, c_p,
                                        c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_pointconv_bwd_scratch_floats": (c_i64, [c_i, c_i, c_i, c_i, c_i]),
    "b200_pointconv_bwd": (c_i, [c_p, c_p, c_p, c_p, ctypes.POINTER(PointConvWeights), c_p, ctypes.POINTER(PointConvGrads),
                                 c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_knn_interpolate": (c_i, [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_knn_interpolate_bwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_corr3d_scratch_floats": (c_i64, [c_i, c_i, c_i, c_i, c_i, c_i]),
    "b200_corr3d_fwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, ctypes.POINTER(Corr3dWeights), c_p, c_p,
                              c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_corr3d_bwd_scratch_floats": (c_i64, [c_i, c_i, c_i, c_i, c_i, c_i]),
    "b200_corr3d_bwd": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, ctypes.POINTER(Corr3dWeights), c_p, c_p,
                              ctypes.POINTER(Corr3dGrads), c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_corr3d_bwd_det_scratch_bytes": (c_i64, [c_i, c_i, c_i, c_i, c_i, c_i]),
    "b200_corr3d_bwd_det": (c_i, [c_p, c_p, c_p, c_p, c_p, c_p, ctypes.POINTER(Corr3dWeights), c_p, c_p,
                                  ctypes.POINTER(Corr3dGrads), c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p]),
    "b200_event_voxel_int": (c_i, [c_p, c_i64, c_p, c_i, c_i, c_i, c_i, c_p, c_p]),
    "b200_event_voxel_trilinear": (c_i, [c_p, c_p, c_p, c_p, c_i64, c_p, c_i, c_i, c_i, c_i, c_p, c_p]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"rpeflow_b200: {LIB_PATH} is missing. This package has no CPU or torch fallback; build the sm_100a "
            f"library first (python __graft_entry__.py, or make -C rpeflow_b200/csrc).")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise ImportError(f"rpeflow_b200: {LIB_PATH} does not export {name}; rebuild it") from e
        fn.restype, fn.argtypes = res, args
    got = lib.b200_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"rpeflow_b200: ABI mismatch, library {got} != bindings {ABI_VERSION}; rebuild it")
    return lib


B200_ENOSUP = -3        # include/b200flow.h
lib = _load()
LAUNCHES = 0          # kernels of this library launched by this process (bench.py reports it as gpu_launches)
KERNELS_PER_CALL = {"b200_knn_grid": 3, "b200_knn_grid_cf": 3, "b200_pointconv_fwd": 2, "b200_pointconv_fwd_linear": 2, "b200_pointconv_bwd": 6, "b200_corr2d_bwd": 2, "b200_project_nn_corr": 2, "b200_corr3d_fwd": 5, "b200_corr3d_bwd": 10, "b200_corr3d_bwd_det": 26, "b200_event_voxel_trilinear": 3,
                    "b200_knn_interpolate_bwd": 1, "b200_backwarp2d_bwd": 1, "b200_corr2d_bwd_nchw": 2, "b200_convex_upsample_bwd": 2, "b200_fps_large": 5,
                    "b200_grid_sample_pts_bwd": 1, "b200_gather_cf_bwd": 1, "b200_gather_cl_bwd": 1}


class B200Error(RuntimeError):
    pass


def check(rc, what):
    """0 -> ok; otherwise raise RuntimeError like the reference's TORCH_CHECK does."""
    global LAUNCHES
    LAUNCHES += KERNELS_PER_CALL.get(what, 1)
    if rc != 0:
        raise B200Error(f"{what} failed ({rc}): {lib.b200_last_error().decode()}")


def require_dense(what, **tensors):
    """Raise unless every tensor is a contiguous CUDA tensor of the dtype the kernels read (int64 for names starting
    with "knn" or "idx", fp32 otherwise): the entry points pass raw data pointers and would read any other layout wrongly."""
    import torch
    for name, t in tensors.items():
        want = torch.int64 if name.startswith(("knn", "idx")) else torch.float32
        if not (t.is_cuda and t.dtype == want and t.is_contiguous()):
            raise ValueError(f"{what}: {name} must be a contiguous CUDA {want} tensor, got {t.dtype} on {t.device}"
                             f"{'' if t.is_contiguous() else ', not contiguous'} (the functional form converts it)")
