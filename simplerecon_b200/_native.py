"""ctypes binding of ``libsrcv_b200.so`` (the C ABI declared in include/srcv_b200.h).

There is NO fallback: if the library is missing, was built for another
architecture, or a call fails, the caller gets an exception.  In particular the
oracle under ``oracle/`` is test infrastructure and is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "lib" / "libsrcv_b200.so"

VARIANT_AUTO, VARIANT_GENERIC, VARIANT_FAST = 0, 1, 2
LAYOUT_NCHW, LAYOUT_CHUNK_PLANAR = 0, 1
PLANES_FROM_RANGE, PLANES_PER_PLANE, PLANES_PER_PIXEL = 0, 1, 2


class NativeLibraryError(RuntimeError):
    pass


class SrcvError(RuntimeError):
    def __init__(self, status: int, what: str):
        super().__init__(f"srcv status {status}: {what}")
        self.status = status


_fp = C.c_void_p  # device pointers travel as plain addresses


class Shape(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("B", "K", "C", "H", "W", "D", "layout")]


class Planes(C.Structure):
    _fields_ = [("mode", C.c_int32), ("planes", _fp), ("min_depth", _fp), ("max_depth", _fp),
                ("ramp", _fp), ("planes_out", _fp), ("range_per_frame", C.c_int32)]


class Cameras(C.Structure):
    _fields_ = [("src_extrinsics", _fp), ("src_poses", _fp), ("src_Ks", _fp), ("cur_invK", _fp),
                ("src_cam_T_world", _fp), ("cur_world_T_cam", _fp), ("cur_cam_T_world", _fp),
                ("src_world_T_cam", _fp)]


class MlpWeights(C.Structure):
    _fields_ = [("w1", _fp), ("b1", _fp), ("w2", _fp), ("b2", _fp), ("w3", _fp), ("b3", _fp),
                ("hidden1", C.c_int32), ("hidden2", C.c_int32), ("packed_image", _fp)]


class MlpGrads(C.Structure):
    _fields_ = [(n, _fp) for n in ("w1", "b1", "w2", "b2", "w3", "b3")]


class TsdfVolume(C.Structure):
    _fields_ = [("tsdf_values", _fp), ("tsdf_weights", _fp), ("X", C.c_int32), ("Y", C.c_int32), ("Z", C.c_int32),
                ("origin", C.c_float * 3), ("voxel_size", C.c_float), ("truncation_voxels", C.c_float),
                ("max_weight", C.c_float)]


class TsdfFrames(C.Structure):
    _fields_ = [("depth", _fp), ("cam_T_world", _fp), ("K", _fp), ("depth_mask", _fp), ("B", C.c_int32),
                ("H", C.c_int32), ("W", C.c_int32), ("min_depth", C.c_float), ("max_depth", C.c_float)]


class MeshVolume(C.Structure):
    _fields_ = [("tsdf_values", _fp), ("X", C.c_int32), ("Y", C.c_int32), ("Z", C.c_int32),
                ("single_mesh", C.c_int32)]


class MvsScan(C.Structure):
    _fields_ = [("depths", _fp), ("K", _fp), ("K_inv", _fp), ("cam_T_world", _fp), ("world_T_cam", _fp),
                ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32)]


class MvLossArgs(C.Structure):
    _fields_ = [(n, _fp) for n in ("depth_pred", "cur_depth", "src_depth", "cur_invK", "src_K", "cur_world_T_cam",
                                   "src_cam_T_world")] + [(n, C.c_int32) for n in ("B", "K", "H", "W")]


# every symbol include/srcv_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "srcv_abi_version": (C.c_int32, []),
    "srcv_check_device": (C.c_int32, []),
    "srcv_status_string": (C.c_char_p, [C.c_int32]),
    "srcv_last_error": (C.c_char_p, []),
    "srcv_dot_workspace_bytes": (C.c_size_t, [C.POINTER(Shape)]),
    "srcv_dot_forward_f32": (C.c_int32, [C.POINTER(Shape), _fp, _fp, C.POINTER(Cameras),
                                         C.POINTER(Planes), _fp, _fp, _fp, C.c_size_t, _fp]),
    "srcv_dot_backward_workspace_bytes": (C.c_size_t, [C.POINTER(Shape)]),
    "srcv_dot_backward_supported": (C.c_int32, [C.POINTER(Shape)]),
    "srcv_dot_backward_f32": (C.c_int32, [C.POINTER(Shape), _fp, _fp, C.POINTER(Cameras), C.POINTER(Planes),
                                          _fp, _fp, _fp, _fp, C.c_size_t, _fp]),
    "srcv_warp_workspace_bytes": (C.c_size_t, [C.POINTER(Shape)]),
    "srcv_warp_features_f32": (C.c_int32, [C.POINTER(Shape), _fp, C.POINTER(Cameras), _fp, C.c_int32,
                                           _fp, _fp, _fp, _fp, C.c_size_t, _fp]),
    "srcv_warp_features_planes_f32": (C.c_int32, [C.POINTER(Shape), _fp, C.POINTER(Cameras), _fp, C.c_int32,
                                                  _fp, _fp, _fp, _fp, _fp, C.c_size_t, _fp]),
    "srcv_mlp_workspace_bytes": (C.c_size_t, [C.POINTER(Shape), C.POINTER(MlpWeights)]),
    "srcv_mlp_packed_bytes": (C.c_size_t, [C.POINTER(Shape), C.POINTER(MlpWeights)]),
    "srcv_mlp_pack_weights": (C.c_int32, [C.POINTER(Shape), C.POINTER(MlpWeights), _fp, _fp]),
    "srcv_mlp_forward_f32": (C.c_int32, [C.POINTER(Shape), _fp, _fp, C.POINTER(Cameras),
                                         C.POINTER(Planes), C.POINTER(MlpWeights), _fp, _fp, _fp,
                                         _fp, C.c_size_t, _fp]),
    "srcv_mlp_backward_workspace_bytes": (C.c_size_t, [C.POINTER(Shape), C.POINTER(MlpWeights)]),
    "srcv_mlp_backward_supported": (C.c_int32, [C.POINTER(Shape), C.c_int32, C.c_int32]),
    "srcv_mlp_backward_f32": (C.c_int32, [C.POINTER(Shape), _fp, _fp, C.POINTER(Cameras), C.POINTER(Planes),
                                          C.POINTER(MlpWeights), _fp, _fp, _fp, C.POINTER(MlpGrads), _fp,
                                          C.c_size_t, _fp]),
    "srcv_instnorm_to_chunk_planar_f32": (C.c_int32, [_fp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                      C.c_float, _fp, _fp, _fp]),
    "srcv_tsdf_workspace_bytes": (C.c_size_t, [C.POINTER(TsdfFrames)]),
    "srcv_tsdf_integrate_f16": (C.c_int32, [C.POINTER(TsdfVolume), C.POINTER(TsdfFrames), _fp, C.c_size_t, _fp]),
    "srcv_mesh_workspace_bytes": (C.c_size_t, [C.POINTER(MeshVolume)]),
    "srcv_mesh_scratch_bytes": (C.c_size_t, [C.c_int32]),
    "srcv_mesh_count_f16": (C.c_int32, [C.POINTER(MeshVolume), _fp, _fp, C.c_size_t, _fp]),
    "srcv_mesh_emit_f16": (C.c_int32, [C.POINTER(MeshVolume), C.c_int32, C.c_int32, _fp, _fp, _fp, _fp, _fp,
                                       C.c_size_t, _fp, C.c_size_t, _fp]),
    "srcv_mvs_workspace_bytes": (C.c_size_t, [C.POINTER(MvsScan)]),
    "srcv_mvs_consistency_f32": (C.c_int32, [C.POINTER(MvsScan), C.c_int32, C.c_float, C.c_int32, _fp, _fp, _fp,
                                             _fp, C.c_size_t, C.c_int32, _fp]),
    "srcv_mvloss_workspace_bytes": (C.c_size_t, [C.POINTER(MvLossArgs)]),
    "srcv_mvloss_forward_f32": (C.c_int32, [C.POINTER(MvLossArgs), _fp, _fp, _fp, _fp, C.c_size_t, _fp]),
    "srcv_mvloss_backward_f32": (C.c_int32, [C.POINTER(MvLossArgs), _fp, _fp, _fp, C.c_size_t, _fp]),
    "srcv_set_variant": (C.c_int32, [C.c_int32]),
    "srcv_last_variant": (C.c_char_p, []),
    "srcv_launch_count": (C.c_uint64, []),
    "srcv_tc_selftest_f32": (C.c_int32, [_fp, _fp, C.c_int32, _fp, _fp, _fp]),
    "srcv_profile_begin": (C.c_int32, [C.c_int32]),
    "srcv_profile_end": (C.c_int32, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
}

_lib = None


def load() -> C.CDLL:
    """Loads the in-tree shared library (built by ``__graft_entry__.build()`` /
    ``python -m simplerecon_b200.build``).  Raises if it is not there."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("SRCV_B200_LIB", LIB_PATH))
    if not path.is_file():
        raise NativeLibraryError(
            f"{path} not found — build it with `python -m simplerecon_b200.build` "
            "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(str(path))
    for name, (res, args) in SYMBOLS.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover
            raise NativeLibraryError(f"{path} does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    if lib.srcv_abi_version() != 2:
        raise NativeLibraryError(f"ABI version mismatch: library {lib.srcv_abi_version()}, binding 2")
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        lib = load()
        what = lib.srcv_last_error().decode() or lib.srcv_status_string(status).decode()
        raise SrcvError(status, what)


def set_variant(v: int) -> None:
    check(load().srcv_set_variant(v))


def last_variant() -> str:
    return load().srcv_last_variant().decode()


def launch_count() -> int:
    return int(load().srcv_launch_count())


def profile_begin(max_records: int) -> None:
    check(load().srcv_profile_begin(max_records))


def profile_end():
    """Returns (prep_ms_total, sweep_ms_total, n_records)."""
    a, b, n = C.c_double(0), C.c_double(0), C.c_int32(0)
    check(load().srcv_profile_end(C.byref(a), C.byref(b), C.byref(n)))
    return a.value, b.value, n.value
