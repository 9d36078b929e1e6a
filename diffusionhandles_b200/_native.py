"""ctypes binding of libdiffhandles_b200.so (include/dh_b200.h).

The library is a plain C-ABI shared object: no torch types cross the boundary, only device pointers
(``tensor.data_ptr()``), sizes and the current CUDA stream handle.  There is NO fallback: if the
library cannot be loaded, or a tensor is not on a CUDA device, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

from . import build as _build

_LIB: Optional[C.CDLL] = None

c_void_p, c_int, c_float, c_size_t = C.c_void_p, C.c_int, C.c_float, C.c_size_t


class NativeLibraryError(RuntimeError):
    """libdiffhandles_b200.so is missing or failed; the product has no CPU / PyTorch fallback."""


class dh_camera(C.Structure):
    _fields_ = [("k", c_float * 9), ("kinv", c_float * 9)]


class dh_rigid(C.Structure):
    _fields_ = [("axis", c_float * 3), ("_pad", c_float), ("cos_t", C.c_double), ("sin_t", C.c_double),
                ("t", C.c_double * 3)]


class dh_warp_level(C.Structure):
    _fields_ = [("inp", c_void_p), ("out", c_void_p), ("src_map", c_void_p), ("channels", C.c_int32), ("hw", C.c_int32)]


class dh_loss_layer(C.Structure):
    _fields_ = [("cur", c_void_p), ("orig", c_void_p), ("grad", c_void_p), ("channels", C.c_int32), ("h", C.c_int32),
                ("w", C.c_int32), ("fg_weight", c_float), ("bg_weight", c_float), ("resize_tables", c_void_p)]


class dh_ddim_coeffs(C.Structure):
    _fields_ = [("guidance_scale", c_float), ("sqrt_beta_t", c_float), ("sqrt_alpha_t", c_float), ("sqrt_alpha_prev", c_float),
                ("sqrt_beta_prev", c_float), ("divide_by_reciprocal", C.c_int32)]


class dh_loss_plan_desc(C.Structure):
    _fields_ = [("n_pairs", C.c_int32), ("box_cells", C.c_int32), ("flags", C.c_int32), ("ell_slices", C.c_int32),
                ("ell_groups", C.c_int32), ("n_src_cells", C.c_int32)]


class dh_loss_batch_edit(C.Structure):
    _fields_ = [("layers", C.POINTER(dh_loss_layer)), ("n_layers", C.c_int32), ("plan", c_void_p), ("desc", dh_loss_plan_desc),
                ("n_fg", C.c_int32), ("n_bg_orig", C.c_int32), ("n_bg_trans", C.c_int32), ("n_bg_common", C.c_int32),
                ("loss_out", c_void_p)]


_SIGNATURES = {
    "dh_status_string": (C.c_char_p, [c_int]),
    "dh_abi_version": (c_int, []),
    "dh_last_cuda_error": (c_int, []),
    "dh_device_info": (c_int, [C.POINTER(c_int)] * 3),
    "dh_linspace_f32_host": (c_int, [c_float, c_float, c_int, C.POINTER(c_float)]),
    "dh_unproject": (c_int, [c_void_p, c_int, c_int, c_int, C.POINTER(dh_camera), c_void_p, c_void_p, c_void_p, c_void_p]),
    "dh_transform_points_workspace_bytes": (c_size_t, [c_int]),
    "dh_transform_points": (c_int, [c_void_p, c_int, c_float, C.POINTER(c_float), C.POINTER(c_float), c_void_p, c_void_p,
                                    c_size_t, c_void_p]),
    "dh_edit_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dh_edit_splat": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, C.POINTER(dh_camera), C.POINTER(dh_rigid), c_void_p,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dh_edit_objects_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dh_edit_splat_objects": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, C.POINTER(dh_camera),
                                      C.POINTER(dh_rigid), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                      c_void_p]),
    "dh_transform_point_cloud_workspace_bytes": (c_size_t, [c_int]),
    "dh_transform_point_cloud": (c_int, [c_void_p, c_void_p, c_int, C.POINTER(dh_rigid), c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_size_t, c_void_p]),
    "dh_project_points": (c_int, [c_void_p, c_int, c_int, c_int, C.POINTER(dh_camera), c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p]),
    "dh_splat_zbuffer": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dh_splat_resolve": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dh_splat_visible": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                 c_void_p, c_void_p]),
    "dh_inv_minmax": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dh_disparity": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dh_morph_pass": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, C.POINTER(C.c_uint32), c_int, c_int, c_int, c_void_p]),
    "dh_mask_clean": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, C.POINTER(C.c_uint32), c_int,
                              C.POINTER(C.c_uint32), c_int, c_void_p]),
    "dh_unpack_bits": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "dh_pack_mask_bits": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dh_correspondences": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                   c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dh_process_correspondences": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p]),
    "dh_dense_source_maps": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, C.POINTER(c_int), c_int, c_void_p, c_void_p]),
    "dh_warp_gather_list": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "dh_warp_gather_dense": (c_int, [C.POINTER(dh_warp_level), c_int, c_int, c_void_p]),
    "dh_guidance_loss_workspace_bytes": (c_size_t, [c_int, c_int]),
    "dh_guidance_loss_patch_workspace_bytes": (c_size_t, [c_int, c_int]),
    "dh_guidance_loss_patch": (c_int, [C.POINTER(dh_loss_layer), c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                       c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dh_guidance_loss_patch_batch_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dh_guidance_loss_patch_batch": (c_int, [C.POINTER(dh_loss_batch_edit), c_int, c_int, c_int, c_int, c_int, c_void_p, c_size_t,
                                             c_void_p]),
    "dh_loss_resize_tables_bytes": (c_size_t, []),
    "dh_build_loss_resize_tables": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dh_loss_plan_bytes": (c_size_t, [c_int, c_int]),
    "dh_loss_plan_workspace_bytes": (c_size_t, [c_int, c_int]),
    "dh_build_loss_plan": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int,
                                   c_void_p, c_size_t, c_void_p, c_size_t, c_void_p]),
    "dh_loss_plan_info": (c_int, [c_void_p, C.POINTER(dh_loss_plan_desc)]),
    "dh_guidance_loss": (c_int, [C.POINTER(dh_loss_layer), c_int, c_int, c_void_p, C.POINTER(dh_loss_plan_desc), c_int, c_int, c_int, c_int,
                                 c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dh_guidance_loss_batch_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dh_guidance_loss_batch": (c_int, [C.POINTER(dh_loss_batch_edit), c_int, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "dh_scale_inplace_many": (c_int, [C.POINTER(c_void_p), C.POINTER(c_size_t), c_int, c_void_p, c_void_p]),
    "dh_latent_step": (c_int, [c_void_p, c_void_p, c_float, c_void_p, c_size_t, c_void_p]),
    "dh_cfg_ddim_step": (c_int, [c_void_p, c_void_p, c_void_p, C.POINTER(dh_ddim_coeffs), c_void_p, c_void_p, c_size_t, c_void_p]),
    "dh_raster_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dh_rasterize_meshes": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, C.POINTER(c_float), C.POINTER(c_float), c_float,
                                    c_float, c_float, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                    c_void_p]),
    "dh_interpolate_face_attributes": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dh_edit_mesh_batch_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "dh_edit_mesh_batch": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int,
                                   C.POINTER(c_float), C.POINTER(c_float), C.POINTER(c_float), c_int, c_int, C.POINTER(c_float),
                                   C.POINTER(c_float), c_float, c_float, c_float, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_size_t, c_void_p]),
    "dh_edit_mesh_scenes_workspace_bytes": (c_size_t, [c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                                       C.POINTER(C.c_int32), c_int, C.POINTER(C.c_int32), c_int, c_int]),
    "dh_edit_mesh_scenes": (c_int, [c_int, c_void_p, c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), c_void_p, c_void_p, c_void_p,
                                    C.POINTER(C.c_int32), C.POINTER(C.c_int32), c_int, C.POINTER(C.c_int32), C.POINTER(c_float),
                                    C.POINTER(c_float), C.POINTER(c_float), c_int, c_int, C.POINTER(c_float), C.POINTER(c_float), c_float,
                                    c_float, c_float, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t,
                                    c_void_p]),
    "dh_poisson_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "dh_poisson_fill": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, C.c_double,
                                c_void_p, c_void_p, c_size_t, c_void_p]),
    "dh_poisson_fill_source": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, C.c_double,
                                       c_void_p, c_void_p, c_size_t, c_void_p]),
}

# symbols include/dh_b200.h declares; tests check that every one of them is exported
DECLARED_SYMBOLS = tuple(_SIGNATURES)


def library_path() -> str:
    return os.environ.get("DH_B200_LIB", _build.LIB_PATH)


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (once) and return the shared library.  Raises NativeLibraryError when that is impossible."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path) or (path == _build.LIB_PATH and not _build.is_current() and _can_build()):
        if not (build_if_missing and _can_build()):
            raise NativeLibraryError(
                f"{path} not found and nvcc is unavailable; build it with `python -m diffusionhandles_b200.build`. "
                "There is no CPU fallback.")
        _build.build()
    try:
        lib = C.CDLL(path)
    except OSError as e:  # pragma: no cover
        raise NativeLibraryError(f"cannot load {path}: {e}") from e
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:
            raise NativeLibraryError(f"{path} does not export {name}") from e
        fn.restype, fn.argtypes = res, args
    if lib.dh_abi_version() != 1:
        raise NativeLibraryError(f"ABI version mismatch: library {lib.dh_abi_version()}, binding 1")
    _LIB = lib
    return lib


def _can_build() -> bool:
    try:
        _build._nvcc()
        return True
    except RuntimeError:
        return False


def check(rc: int, what: str = "") -> None:
    if rc == 0:
        return
    lib = load()
    msg = lib.dh_status_string(rc).decode()
    if rc == -3:
        msg += f" (cudaError {lib.dh_last_cuda_error()})"
    if rc == -1:
        raise ValueError(f"libdiffhandles_b200 {what}: {msg}")
    raise RuntimeError(f"libdiffhandles_b200 {what}: {msg}")


def ptr(t: Optional[torch.Tensor], dtype: Optional[torch.dtype] = None, name: str = "tensor") -> Optional[int]:
    """Device pointer of a contiguous CUDA tensor (or None)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeLibraryError(f"{name} must live on a CUDA device (got {t.device}); there is no CPU path")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name} must be {dtype}, got {t.dtype}")
    return t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_handle(device: torch.device) -> int:
    """cudaStream_t of torch's current stream on ``device`` (the raw getter avoids building a Stream object per call)."""
    cur = torch.cuda.current_device()
    idx = cur if device.index is None else device.index
    if idx != cur:
        # the C ABI launches on the CURRENT device; a tensor that lives elsewhere would be dereferenced on the wrong GPU
        raise NativeLibraryError(f"tensors are on cuda:{idx} but the current CUDA device is cuda:{cur}; "
                                 f"run the call under `with torch.cuda.device({idx}):` (one process per GPU is the intended use)")
    if _raw_stream is not None:
        return _raw_stream(idx)
    return torch.cuda.current_stream(device).cuda_stream


def make_camera(intrinsics: torch.Tensor) -> dh_camera:
    """dh_camera from a (3,3) fp32 intrinsics tensor; the inverse is torch.linalg.inv on the CPU in fp32,
    exactly what depth_transform.py:595 computes."""
    K = intrinsics.detach().to(device="cpu", dtype=torch.float32).contiguous()
    Kinv = torch.linalg.inv(K).contiguous()
    cam = dh_camera()
    cam.k[:] = K.reshape(-1).tolist()
    cam.kinv[:] = Kinv.reshape(-1).tolist()
    return cam


def u32_array(values):
    return (C.c_uint32 * len(values))(*[int(v) for v in values])
