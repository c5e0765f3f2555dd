"""ctypes binding of libmkb200.so (include/mkb200.h).  No CPU fallback: if the CUDA library is missing or
no CUDA device is present, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "lib", "libmkb200.so")

MKB_OK = 0
OCC_ACCUMULATE = 1
OCC_LAYOUT_CXYZ = 2
DIST_DISTANCES = 0
DIST_CONTACTS = 1
DIST_DISTANCES_FAST = 4

# numpy mirror of `mkb_grid_desc` (72 bytes, no padding)
GRID_DESC = np.dtype(
    [("origin", "<f8", (3,)), ("voxelsize", "<f8"), ("dims", "<i4", (3,)), ("reserved", "<i4"),
     ("atom_begin", "<i8"), ("atom_end", "<i8"), ("out_offset", "<i8")], align=False)
assert GRID_DESC.itemsize == 72


class Traj(C.Structure):
    """mirror of `mkb_traj`"""
    _fields_ = [("coords", C.c_void_p), ("box", C.c_void_p), ("n_atoms", C.c_int64), ("n_frames", C.c_int64),
                ("frame_stride", C.c_int64), ("frame_stride_box", C.c_int64)]


EXPORTS = [
    "mkb_version", "mkb_create", "mkb_destroy", "mkb_last_error", "mkb_launch_count",
    "mkb_set_timing", "mkb_get_timing", "mkb_last_kernel",
    "mkb_occupancy_grid_batch_compact", "mkb_occupancy_compact_blocks", "mkb_occupancy_expand_host",
    "mkb_occupancy_grid_batch_to_host", "mkb_occupancy_wait_index",
    "mkb_occupancy_grid_batch", "mkb_occupancy_grid_batch_masked", "mkb_occupancy_points",
    "mkb_grid_centers", "mkb_rotate_coords",
    "mkb_dist_trajectory", "mkb_contacts_count", "mkb_contacts_fill", "mkb_dist_reduction",
    "mkb_cdist", "mkb_pdist", "mkb_squareform", "mkb_collisions_count", "mkb_collisions_fill",
    "mkb_bonds_count", "mkb_bonds_fill", "mkb_shell_counts", "mkb_wrap_box", "mkb_within_distance", "mkb_xtc_decode",
    "mkb_wrap_triclinic", "mkb_hbonds_count", "mkb_hbonds_fill", "mkb_ring_pairs_count", "mkb_ring_pairs_fill",
    "mkb_align_fit", "mkb_align_apply", "mkb_rmsd",
]

_lib = None
_handles: dict[int, C.c_void_p] = {}


class MkbError(RuntimeError):
    pass


class MkbUnsupported(MkbError):
    """MKB_ERR_UNSUPPORTED: a valid request outside the domain of the entry point (callers fall back to the general one)."""


def load():
    """dlopen the library (works without a GPU; creating a handle does not)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("MKB200_LIB", LIB_PATH)  # tuning hook: an alternative in-tree build of the same sources
    if not os.path.isfile(path):
        raise ImportError(
            f"{path} not found: build the CUDA extension first (python -m moleculekit_b200.build). "
            "moleculekit_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    vp, i32, i64, u32, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_float
    lib.mkb_version.restype = C.c_int
    lib.mkb_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.mkb_destroy.argtypes = [vp]
    lib.mkb_last_error.argtypes = [vp]
    lib.mkb_last_error.restype = C.c_char_p
    lib.mkb_launch_count.argtypes = [vp]
    lib.mkb_launch_count.restype = i64
    lib.mkb_set_timing.argtypes = [vp, C.c_int]
    lib.mkb_get_timing.argtypes = [vp, C.POINTER(f32), C.POINTER(f32)]
    lib.mkb_last_kernel.argtypes = [vp]
    lib.mkb_last_kernel.restype = C.c_char_p
    lib.mkb_occupancy_grid_batch.argtypes = [vp, vp, vp, vp, i64, i32, vp, i32, vp, u32]
    lib.mkb_occupancy_grid_batch_compact.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, i32, vp, vp, i64]
    lib.mkb_occupancy_grid_batch_to_host.argtypes = [vp, vp, vp, vp, vp, vp, i64, vp, i32, vp, vp, i64, vp]
    lib.mkb_occupancy_wait_index.argtypes = [vp]
    lib.mkb_occupancy_compact_blocks.argtypes = [vp, i32]
    lib.mkb_occupancy_compact_blocks.restype = i64
    lib.mkb_occupancy_expand_host.argtypes = [vp, i32, i32, vp, vp, i64, vp, i32, i32]
    lib.mkb_occupancy_points.argtypes = [vp, vp, vp, i64, vp, vp, i64, i32, vp, u32]
    lib.mkb_occupancy_grid_batch_masked.argtypes = [vp, vp, vp, vp, vp, i64, i32, vp, i32, vp, u32]
    lib.mkb_grid_centers.argtypes = [vp, vp, vp, i32, vp]
    lib.mkb_rotate_coords.argtypes = [vp, vp, vp, i64, vp, i32, vp, vp, vp, vp]
    tp = C.POINTER(Traj)
    lib.mkb_dist_trajectory.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, i32, i32, i32, f32, f32, vp]
    lib.mkb_contacts_count.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, i32, i32, f32, vp, C.POINTER(i64)]
    lib.mkb_contacts_fill.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, i32, i32, f32, vp, vp]
    lib.mkb_dist_reduction.argtypes = [vp, vp, tp, vp, vp, i64, vp, vp, i64, vp, vp, i32, i32, vp, i32, i32, i32,
                                       i32, f32, f32, vp]
    lib.mkb_cdist.argtypes = [vp, vp, vp, i64, vp, i64, i32, vp]
    lib.mkb_pdist.argtypes = [vp, vp, vp, i64, i32, vp]
    lib.mkb_squareform.argtypes = [vp, vp, vp, i64, i64, vp]
    lib.mkb_collisions_count.argtypes = [vp, vp, vp, i64, vp, i64, f32, vp, C.POINTER(i64)]
    lib.mkb_collisions_fill.argtypes = [vp, vp, vp, i64, vp, i64, f32, vp, vp]
    lib.mkb_shell_counts.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, i32, i32, f32, vp, i32, vp]
    lib.mkb_bonds_count.argtypes = [vp, vp, vp, vp, vp, i64, f32, vp, C.POINTER(i64)]
    lib.mkb_bonds_fill.argtypes = [vp, vp, vp, vp, vp, i64, f32, vp, vp]
    lib.mkb_within_distance.argtypes = [vp, vp, vp, i64, vp, i64, vp, i64, f32, vp]
    lib.mkb_xtc_decode.argtypes = [vp, vp, vp, i64, vp, i64, i64, vp, i64, f32, vp]
    lib.mkb_wrap_box.argtypes = [vp, vp, tp, vp, i64, vp, i64, C.POINTER(C.c_float)]
    lib.mkb_wrap_triclinic.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, i64, C.POINTER(C.c_float), i32]
    lib.mkb_hbonds_count.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, vp, f32, f32, i32, i32, vp, C.POINTER(i64)]
    lib.mkb_hbonds_fill.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, vp, f32, f32, i32, i32, vp, vp]
    lib.mkb_ring_pairs_count.argtypes = [vp, vp, i32, tp, vp, vp, i64, vp, i64, f32, f32, f32, f32, vp, C.POINTER(i64)]
    lib.mkb_ring_pairs_fill.argtypes = [vp, vp, i32, tp, vp, vp, i64, vp, i64, f32, f32, f32, f32, vp, vp, vp]
    lib.mkb_align_fit.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, i64, i32, vp]
    lib.mkb_align_apply.argtypes = [vp, vp, tp, vp, i64, vp]
    lib.mkb_rmsd.argtypes = [vp, vp, tp, vp, i64, vp, i64, vp, i64, i64, vp, vp]
    for name in EXPORTS:
        if name in ("mkb_last_error", "mkb_launch_count", "mkb_version", "mkb_last_kernel", "mkb_occupancy_compact_blocks"):
            continue
        getattr(lib, name).restype = C.c_int
    _lib = lib
    return lib


def handle(device: int = 0):
    """One engine handle per CUDA device, created on first use."""
    lib = load()
    device = int(device)
    h = _handles.get(device)
    if h is None:
        out = C.c_void_p()
        rc = lib.mkb_create(device, C.byref(out))
        if rc != MKB_OK or not out.value:
            raise MkbError(
                f"mkb_create(device={device}) failed (status {rc}): a CUDA device is required, there is no CPU fallback")
        h = out
        _handles[device] = h
    return h


def check(rc: int, h) -> None:
    if rc != MKB_OK:
        msg = load().mkb_last_error(h)
        raise (MkbUnsupported if rc == -5 else MkbError)(f"libmkb200 status {rc}: {msg.decode() if msg else '?'}")


def launch_count(device: int = 0) -> int:
    return int(load().mkb_launch_count(handle(device)))


def set_timing(on: bool, device: int = 0) -> None:
    h = handle(device)
    check(load().mkb_set_timing(h, 1 if on else 0), h)


def get_timing(device: int = 0) -> tuple[float, float]:
    """(prep_ms, main_kernel_ms) of the most recent timed entry point on this device (synchronises)."""
    h = handle(device)
    a, b = C.c_float(), C.c_float()
    check(load().mkb_get_timing(h, C.byref(a), C.byref(b)), h)
    return float(a.value), float(b.value)


def last_fill_kernel(device: int = 0) -> str:
    """Name of the main kernel the most recent occupancy / distance call launched on this device."""
    return load().mkb_last_kernel(handle(device)).decode()


def destroy_all() -> None:
    for dev, h in list(_handles.items()):
        load().mkb_destroy(h)
        del _handles[dev]
