"""visibility_heuristic_path_planner_b200 -- ctypes binding of libvhp_b200.so.

The product is the C-ABI in include/vhp.h (CUDA kernels for sm_100a + C++ host
boundary).  This module is only the thin Python view of it used by tests/ and
bench.py: numpy arrays go through the host-buffer entry points, torch CUDA
tensors through the *_dev entry points (pointers via .data_ptr(), the context
enqueues on torch's current stream).

There is no CPU fallback: `Context()` raises when the library is missing or no
sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "lib", "libvhp_b200.so")
# kernel-tuning experiments only (tools/build_variant.py): load another build of the same library
if os.environ.get("VHP_LIB_VARIANT"):
    LIB_PATH = os.path.join(PKG, "lib_" + os.environ["VHP_LIB_VARIANT"], "libvhp_b200.so")

F32, F64 = 0, 1
RANGE_BOX, RANGE_DISK = 0, 1
NO_PARENT = -1
STATUS_NAMES = {0: "OK", 1: "START_OOB", 2: "END_OOB", 3: "START_OCCUPIED",
                4: "END_OCCUPIED", 5: "MAX_ITER", -1: "ERR_INVALID_ARG",
                -2: "ERR_NO_DEVICE", -3: "ERR_CUDA", -4: "ERR_IO", -5: "ERR_UNSUPPORTED"}


class VhpError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {msg}")
        self.status = status


class PlannerOut(C.Structure):
    _fields_ = [("status", C.c_void_p), ("nb_sources", C.c_void_p),
                ("light_sources", C.c_void_p), ("path_len", C.c_void_p),
                ("path_n", C.c_void_p), ("path", C.c_void_p), ("vg", C.c_void_p),
                ("came", C.c_void_p), ("vis", C.c_void_p)]


class MergeOut(C.Structure):
    """struct vhp_merge_out: vmax (dtype), first (int32), count (uint32), each [group][ny][nx] or NULL."""
    _fields_ = [("vmax", C.c_void_p), ("first", C.c_void_p), ("count", C.c_void_p)]


class CoverOut(C.Structure):
    """struct vhp_cover_out: pick (int32 [prob][k]), gain (uint32 [prob][k]), npicked (int32 [prob]), covered
    (uint32 [prob][ny][ceil(nx/32)]), each may be NULL."""
    _fields_ = [("pick", C.c_void_p), ("gain", C.c_void_p), ("npicked", C.c_void_p), ("covered", C.c_void_p)]


class CoverWeightedOut(C.Structure):
    """struct vhp_cover_weighted_out: pick (int32 [prob][k]), gain (uint64 [prob][k]), npicked (int32 [prob]),
    covered (uint32 [prob][ny][ceil(nx/32)]), each may be NULL."""
    _fields_ = [("pick", C.c_void_p), ("gain", C.c_void_p), ("npicked", C.c_void_p), ("covered", C.c_void_p)]


class CoverMfoldOut(C.Structure):
    """struct vhp_cover_mfold_out: pick (int32 [prob][k]), gain (uint64 [prob][k]), npicked (int32 [prob]), count
    (uint8 [prob][ny][nx]), each may be NULL."""
    _fields_ = [("pick", C.c_void_p), ("gain", C.c_void_p), ("npicked", C.c_void_p), ("count", C.c_void_p)]


class SweepVariant(C.Structure):
    """struct vhp_sweep_variant: model 1 = getAccessibilityMap.m (alpha, fac, light_strength),
    model 2 = computeVisibilityUsingQueue as an order-free rule (cutoff)."""
    _fields_ = [("model", C.c_int32), ("alpha", C.c_double), ("fac", C.c_double),
                ("light_strength", C.c_double), ("cutoff", C.c_double)]


VARIANT_MATLAB, VARIANT_QUEUE = 1, 2


class Config(C.Structure):
    """struct vhp_config (mirror of the reference's struct Config)."""
    _fields_ = [("mode", C.c_int32), ("ncols", C.c_int64), ("nrows", C.c_int64),
                ("nb_of_obstacles", C.c_int64), ("min_width", C.c_int64),
                ("max_width", C.c_int64), ("min_height", C.c_int64),
                ("max_height", C.c_int64), ("random_seed", C.c_int32),
                ("seed_value", C.c_int32), ("image_path", C.c_char * 1024),
                ("start_x", C.c_int32), ("start_y", C.c_int32), ("end_x", C.c_int32),
                ("end_y", C.c_int32), ("max_iter", C.c_int64),
                ("visibility_threshold", C.c_double), ("light_strength", C.c_float),
                ("timer", C.c_int32), ("save_results", C.c_int32),
                ("save_local_visibility", C.c_int32), ("save_came_from", C.c_int32),
                ("save_light_sources", C.c_int32), ("save_global_visibility", C.c_int32),
                ("save_visibility_field", C.c_int32), ("silent", C.c_int32),
                ("ball_radius", C.c_int32)]


_lib = None


def load_library(build_if_missing: bool = True):
    """dlopen libvhp_b200.so (building it in-tree first if it is absent)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise FileNotFoundError(LIB_PATH)
        from .build import build
        build()
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    lib.vhp_abi_version.restype = C.c_int
    lib.vhp_version_string.restype = C.c_char_p
    lib.vhp_device_count.restype = C.c_int
    lib.vhp_context_create.argtypes = [i32, vp, C.POINTER(vp)]
    lib.vhp_context_destroy.argtypes = [vp]
    lib.vhp_context_destroy.restype = None
    lib.vhp_context_synchronize.argtypes = [vp]
    lib.vhp_last_error.argtypes = [vp]
    lib.vhp_last_error.restype = C.c_char_p
    lib.vhp_launch_count.argtypes = [vp]
    lib.vhp_launch_count.restype = i64
    batch = [vp, vp, i32, i32, i32, vp, vp, i64, i32, vp]
    for name in ("vhp_visibility_batch", "vhp_visibility_batch_dev", "vhp_raycast_batch",
                 "vhp_raycast_batch_dev"):
        getattr(lib, name).argtypes = batch
    lib.vhp_visibility_batch_bin.argtypes = [vp, vp, i32, i32, i32, vp, vp, i64, C.c_double, vp]
    lib.vhp_visibility_batch_bin_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, i64, C.c_double, vp]
    lib.vhp_visibility_variant_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, i64, C.POINTER(SweepVariant), i32, vp]
    lib.vhp_visibility_variant_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, i64, C.POINTER(SweepVariant), i32, vp]
    lib.vhp_visibility_batch_runs.argtypes = [vp, vp, i32, i32, i32, vp, vp, i64, C.c_double, vp, vp, vp, i64,
                                              C.POINTER(i64)]
    lib.vhp_runs_to_bits.argtypes = [vp, vp, vp, i64, i32, i32, vp]
    lib.vhp_visibility_merge_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, C.c_double, i32,
                                               C.POINTER(MergeOut)]
    lib.vhp_visibility_merge_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, i64, C.c_double, i32,
                                                   C.POINTER(MergeOut)]
    lib.vhp_visibility_merge_range_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, C.c_int32, C.c_int32,
                                                     C.c_double, i32, C.POINTER(MergeOut)]
    lib.vhp_visibility_merge_range_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, i64, C.c_int32,
                                                         C.c_int32, C.c_double, i32, C.POINTER(MergeOut)]
    lib.vhp_visibility_merge_view_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp, i64, C.c_int32, C.c_int32,
                                                    C.c_double, i32, C.POINTER(MergeOut)]
    lib.vhp_visibility_merge_view_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp, i64, i64, C.c_int32,
                                                        C.c_int32, C.c_double, i32, C.POINTER(MergeOut)]
    lib.vhp_visibility_cover_greedy_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, C.c_int32, C.c_int32,
                                                      C.c_int32, C.c_double, vp, C.POINTER(CoverOut)]
    lib.vhp_visibility_cover_greedy_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, i64, C.c_int32,
                                                          C.c_int32, C.c_int32, C.c_double, vp, C.POINTER(CoverOut)]
    lib.vhp_visibility_cover_greedy_weighted_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, C.c_int32,
                                                               C.c_int32, C.c_int32, C.c_double, vp,
                                                               C.POINTER(CoverWeightedOut)]
    lib.vhp_visibility_cover_greedy_weighted_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, i64,
                                                                   C.c_int32, C.c_int32, C.c_int32, C.c_double, vp,
                                                                   C.POINTER(CoverWeightedOut)]
    lib.vhp_visibility_cover_greedy_mfold_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, C.c_int32,
                                                            C.c_int32, C.c_int32, C.c_double, vp, C.c_int32,
                                                            C.POINTER(CoverMfoldOut)]
    lib.vhp_visibility_cover_greedy_mfold_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, i64, i64,
                                                                C.c_int32, C.c_int32, C.c_int32, C.c_double, vp,
                                                                C.c_int32, C.POINTER(CoverMfoldOut)]
    lib.vhp_visibility_cover_greedy_view_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp, i64, C.c_int32,
                                                           C.c_int32, C.c_int32, C.c_double, vp, C.c_int32,
                                                           C.POINTER(CoverMfoldOut)]
    lib.vhp_visibility_cover_greedy_view_batch_dev.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, vp, i64, i64,
                                                               C.c_int32, C.c_int32, C.c_int32, C.c_double, vp,
                                                               C.c_int32, C.POINTER(CoverMfoldOut)]
    for name in ("vhp_visibility_window_batch", "vhp_visibility_window_batch_dev"):
        getattr(lib, name).argtypes = [vp, vp, i32, i32, i32, vp, vp, i64, C.c_int32, i32, vp]
    lib.vhp_visibility_batch_packed.argtypes = [vp, vp, i32, i32, i32, vp, vp, i64, i32, C.POINTER(vp)]
    for name in ("vhp_packed_pairs", "vhp_packed_bytes", "vhp_packed_pair_bytes"):
        getattr(lib, name).argtypes = [vp]
        getattr(lib, name).restype = i64
    lib.vhp_packed_expand.argtypes = [vp, i64, i64, vp, i32]
    lib.vhp_packed_destroy.argtypes = [vp]
    lib.vhp_packed_destroy.restype = None
    lib.vhp_release_maps_dev.argtypes = [vp]
    lib.vhp_context_device.argtypes = [vp]
    lib.vhp_prepare_maps_dev.argtypes = [vp, vp, i32, i32, i32]
    plan = [vp, vp, i32, i32, i32, vp, vp, i64, C.c_double, C.c_int32, C.c_int32, i32,
            C.POINTER(PlannerOut)]
    lib.vhp_planner_batch.argtypes = plan
    lib.vhp_planner_batch_dev.argtypes = plan
    lib.vhp_strip_halo_rows.argtypes = [i32, i32, i32, i32, i32, i32, C.POINTER(C.c_int32 * 4)]
    lib.vhp_strip_halo_rows.restype = None
    lib.vhp_context_set_grid_sweep.argtypes = [vp, i32]
    lib.vhp_context_set_result_transport.argtypes = [vp, i32]
    lib.vhp_context_set_result_gpu_share.argtypes = [vp, i32]
    lib.vhp_expand_packed_chunk.argtypes = [vp, vp, vp, i32, vp, i64, i64, vp, i32]
    lib.vhp_expand_packed_range.argtypes = [vp, vp, vp, i32, vp, i64, i64, i64, i64, vp]
    lib.vhp_context_last_transport.argtypes = [vp, C.POINTER(i64), C.POINTER(i64),
                                               C.POINTER(C.c_int32)]
    lib.vhp_environment_draw.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint32]
    lib.vhp_environment_draw.restype = C.c_uint32
    lib.vhp_environment_generate_batch_dev.argtypes = [vp, vp, C.c_uint64, i64, i32, vp]
    lib.vhp_strip_sweep_dev.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, C.POINTER(vp * 4), i32, vp]
    lib.vhp_strip_epilogue_dev.argtypes = [vp, i32, i32, i32, i32, i32, i32, i32, i32, C.c_double,
                                           C.c_int32, vp, vp, vp, vp, vp, vp]
    lib.vhp_giant_unique_id.argtypes = [vp]
    lib.vhp_giant_create.argtypes = [vp, vp, i32, i32, i32, i32, vp, i32, C.POINTER(vp)]
    lib.vhp_giant_destroy.argtypes = [vp]
    lib.vhp_giant_destroy.restype = None
    lib.vhp_giant_strip_bounds.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32)]
    lib.vhp_giant_local_rows.argtypes = [vp, C.POINTER(i32), C.POINTER(i32)]
    lib.vhp_giant_set_loop_mode.argtypes = [vp, i32, i32]
    lib.vhp_giant_solve.argtypes = [vp, vp, C.c_double, C.c_int32, C.c_int32, i32, C.POINTER(PlannerOut), vp]
    lib.vhp_context_set_planner_loop.argtypes = [vp, i32]
    lib.vhp_selftest_ratio.argtypes = [vp, i32, C.POINTER(i64)]
    lib.vhp_export_came_from_u64.argtypes = [vp, i64, vp]
    lib.vhp_export_came_from_u64.restype = None
    _lib = lib
    return lib


def _np_ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _cover_weights(weights, shape):
    """weights of the weighted cover calls: None, or uint8 of the problems' (nprob, ny, nx)."""
    if weights is None:
        return None
    w = np.asarray(weights)
    if w.dtype != np.uint8 or w.shape != shape:
        raise ValueError(f"weights must be uint8 of shape {shape}, got {w.dtype} {w.shape}")
    return np.ascontiguousarray(w)


def _occ_u8(occ):
    """(ny, nx) or (nmaps, ny, nx) -> contiguous uint8 (1 free / 0 occupied)."""
    occ = np.asarray(occ)
    if occ.ndim == 2:
        occ = occ[None]
    return np.ascontiguousarray(occ != 0, dtype=np.uint8)


class PackedFields:
    """Handle of vhp_visibility_batch_packed: the fields of a batch in packed form on the host."""

    def __init__(self, lib):
        self.lib, self.h, self.shape, self.dtype = lib, C.c_void_p(), None, None

    def __len__(self):
        return int(self.lib.vhp_packed_pairs(self.h))

    @property
    def nbytes(self):
        """bytes of packed data held (what crossed PCIe)"""
        return int(self.lib.vhp_packed_bytes(self.h))

    def expand(self, first=0, count=None, out=None, threads=0):
        """(count, ny, nx) fields of pairs [first, first + count), bit-identical to visibility_batch."""
        count = len(self) - first if count is None else count
        if out is None:
            out = np.empty((count,) + self.shape, self.dtype)
        st = self.lib.vhp_packed_expand(self.h, first, count, _np_ptr(out), threads)
        if st != 0:
            raise VhpError(st, self.lib.vhp_last_error(None).decode())
        return out

    def close(self):
        if self.h:
            self.lib.vhp_packed_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One device + stream + workspace (vhp_context)."""

    def __init__(self, device: int = 0, stream=None):
        self.lib = load_library()
        h = C.c_void_p()
        st = self.lib.vhp_context_create(int(device), stream, C.byref(h))
        if st != 0:
            raise VhpError(st, self.lib.vhp_last_error(None).decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.lib.vhp_context_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st):
        if st < 0:
            raise VhpError(st, self.lib.vhp_last_error(self.h).decode())
        return st

    def set_grid_sweep(self, mode: int):
        """0: strip sweeps / large planner problems always on one CTA; 1: spread over many CTAs
        by size (default); 2: always (tests)."""
        self._check(self.lib.vhp_context_set_grid_sweep(self.h, int(mode)))

    def set_planner_loop(self, mode: int):
        """How vhp_planner_batch drives a single large problem: 0 automatic (CUDA-graph WHILE
        node), 2 batches of iterations, 3 one host read-back per iteration."""
        self._check(self.lib.vhp_context_set_planner_loop(self.h, int(mode)))

    def set_result_transport(self, mode: int):
        """Transport of host-buffer results: 0 plain copies, 1 automatic (default), 2 always
        packed (uniform / literal 128-byte units, expanded by host threads)."""
        self._check(self.lib.vhp_context_set_result_transport(self.h, int(mode)))

    def set_result_gpu_share(self, sixteenths: int):
        """Packed transport into pinned memory: share of the result (in sixteenths) the GPU
        delivers completely (uniform units included); default 0."""
        self._check(self.lib.vhp_context_set_result_gpu_share(self.h, int(sixteenths)))

    def last_transport(self):
        """(bytes moved device-to-host, bytes of results delivered, transport) of the last
        host-buffer sweep / ray-casting call; transport 0 = plain copies, 1 = packed with a
        staged literal stream, 2 = packed with literal units stored straight into a pinned
        caller buffer."""
        d2h, res, packed = C.c_int64(0), C.c_int64(0), C.c_int32(0)
        self._check(self.lib.vhp_context_last_transport(self.h, C.byref(d2h), C.byref(res),
                                                        C.byref(packed)))
        return int(d2h.value), int(res.value), int(packed.value)

    def synchronize(self):
        self._check(self.lib.vhp_context_synchronize(self.h))

    @property
    def launches(self) -> int:
        return int(self.lib.vhp_launch_count(self.h))

    def selftest_ratio(self, kmax: int) -> int:
        bad = C.c_int64(-1)
        self._check(self.lib.vhp_selftest_ratio(self.h, int(kmax), C.byref(bad)))
        return bad.value

    # ---- host (numpy) entry points ------------------------------------------
    def _batch_host(self, fn, occ, src_xy, src_map, dtype, out=None, pair_shape=None):
        """pair_shape: the result of one pair, (ny, nx) by default."""
        occ = _occ_u8(occ)
        nmaps, ny, nx = occ.shape
        xy = np.ascontiguousarray(src_xy, dtype=np.int32).reshape(-1, 2)
        n = xy.shape[0]
        mp = None if src_map is None else np.ascontiguousarray(src_map, dtype=np.int32)
        odt = np.float32 if dtype == F32 else np.float64
        shape = (n,) + (tuple(pair_shape) if pair_shape is not None else (ny, nx))
        if out is None:
            out = np.empty(shape, dtype=odt)
        elif out.dtype != odt or out.shape != shape or not out.flags.c_contiguous:
            raise ValueError(f"out must be a C-contiguous {shape} array of the result dtype")
        self._check(fn(self.h, _np_ptr(occ), nmaps, nx, ny, _np_ptr(xy), _np_ptr(mp), n,
                       dtype, _np_ptr(out)))
        return out

    def visibility_batch(self, occ, src_xy, src_map=None, dtype=F64, out=None):
        """computeVisibility for every (map, source) pair -> (npairs, ny, nx).  `out`: an
        array to fill instead of a new one (pinned host memory gets the fastest transport)."""
        return self._batch_host(self.lib.vhp_visibility_batch, occ, src_xy, src_map, dtype, out)

    def visibility_window_batch(self, occ, src_xy, radius, src_map=None, dtype=F64, out=None):
        """Range-limited visibility (vhp_visibility_window_batch) -> (npairs, 2R+1, 2R+1): the window of
        visibility_batch's field centred on each source, 0 where it leaves the grid."""
        r = int(radius)
        w = 2 * r + 1 if r >= 0 else 1  # (a negative radius is rejected by the library)

        def fn(h, occ_p, nmaps, nx, ny, xy_p, mp_p, n, dt, out_p):
            return self.lib.vhp_visibility_window_batch(h, occ_p, nmaps, nx, ny, xy_p, mp_p, n, r, dt, out_p)
        return self._batch_host(fn, occ, src_xy, src_map, dtype, out, pair_shape=(w, w))

    def visibility_batch_packed(self, occ, src_xy, src_map=None, dtype=F64, handle=None):
        """computeVisibility for every pair, kept as a lossless packed handle
        (vhp_visibility_batch_packed); `handle`: a PackedFields of an earlier call to refill."""
        occ = _occ_u8(occ)
        nmaps, ny, nx = occ.shape
        xy = np.ascontiguousarray(src_xy, dtype=np.int32).reshape(-1, 2)
        mp = None if src_map is None else np.ascontiguousarray(src_map, dtype=np.int32)
        h = handle if handle is not None else PackedFields(self.lib)
        self._check(self.lib.vhp_visibility_batch_packed(self.h, _np_ptr(occ), nmaps, nx, ny, _np_ptr(xy), _np_ptr(mp),
                                                         xy.shape[0], dtype, C.byref(h.h)))
        h.shape, h.dtype = (ny, nx), (np.float32 if dtype == F32 else np.float64)
        return h

    def visibility_batch_bin(self, occ, src_xy, threshold, src_map=None, out=None):
        """Thresholded binary visibility, bit-packed (vhp_visibility_batch_bin): uint32
        (npairs, ny, ceil(nx/32)), bit b of word w = visibility(32w + b, y) >= threshold."""
        occ = _occ_u8(occ)
        nmaps, ny, nx = occ.shape
        xy = np.ascontiguousarray(src_xy, dtype=np.int32).reshape(-1, 2)
        n = xy.shape[0]
        mp = None if src_map is None else np.ascontiguousarray(src_map, dtype=np.int32)
        wpr = (nx + 31) // 32
        if out is None:
            out = np.empty((n, ny, wpr), dtype=np.uint32)
        elif out.dtype != np.uint32 or out.shape != (n, ny, wpr) or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous uint32 (npairs, ny, ceil(nx/32)) array")
        self._check(self.lib.vhp_visibility_batch_bin(self.h, _np_ptr(occ), nmaps, nx, ny, _np_ptr(xy),
                                                      _np_ptr(mp), n, float(threshold), _np_ptr(out)))
        return out

    def visibility_batch_runs(self, occ, src_xy, threshold, src_map=None, trans_cap=None, out=None):
        """Thresholded visibility as row runs (vhp_visibility_batch_runs).  Returns (row_count uint16
        (npairs, ny), pair_ptr uint64 (npairs + 1), trans uint16 (total,)).  `out` = (row_count, pair_ptr,
        trans) buffers to fill (e.g. pinned); the call is repeated with a larger buffer when the first
        guess for trans is too small and no buffer was given."""
        occ = _occ_u8(occ)
        nmaps, ny, nx = occ.shape
        xy = np.ascontiguousarray(src_xy, dtype=np.int32).reshape(-1, 2)
        n = xy.shape[0]
        mp = None if src_map is None else np.ascontiguousarray(src_map, dtype=np.int32)
        if out is not None:
            rc, pp, tr = out
        else:
            rc = np.empty((n, ny), np.uint16)
            pp = np.empty(n + 1, np.uint64)
            tr = np.empty(int(trans_cap) if trans_cap else max(1024, 16 * n * ny), np.uint16)
        used = C.c_int64(0)
        while True:
            st = self.lib.vhp_visibility_batch_runs(self.h, _np_ptr(occ), nmaps, nx, ny, _np_ptr(xy), _np_ptr(mp), n,
                                                    float(threshold), _np_ptr(rc), _np_ptr(pp), _np_ptr(tr), tr.size,
                                                    C.byref(used))
            if st == -1 and used.value > tr.size and out is None:
                tr = np.empty(max(2 * tr.size, 2 * used.value), np.uint16)
                continue
            self._check(st)
            break
        return rc, pp, tr[: int(pp[n])]

    def visibility_batch_bin_dev(self, occ_t, src_xy_t, threshold, out_bits_t, src_map_t=None):
        nmaps, ny, nx = occ_t.shape
        self._check(self.lib.vhp_visibility_batch_bin_dev(
            self.h, occ_t.data_ptr(), nmaps, nx, ny, src_xy_t.data_ptr(),
            None if src_map_t is None else src_map_t.data_ptr(), src_xy_t.shape[0], float(threshold),
            out_bits_t.data_ptr()))

    def visibility_merge_batch(self, occ, src_xy, group_ptr, threshold, group_map=None, dtype=F64,
                               outputs=("vmax", "first", "count")):
        """Merged visibility of groups of sources (vhp_visibility_merge_batch): group g = sources
        src_xy[group_ptr[g]:group_ptr[g + 1]] on map group_map[g].  Returns a dict of the requested
        outputs, (ngroups, ny, nx) each: vmax (max of the fields, dtype), first (int32, index within
        the group of the first source whose sweep writes the cell with a value >= threshold, NO_PARENT
        if none) and count (uint32, how many do)."""
        return self._merge_host(self.lib.vhp_visibility_merge_batch, (), occ, src_xy, group_ptr, threshold, group_map,
                                dtype, outputs)

    def visibility_merge_range_batch(self, occ, src_xy, group_ptr, threshold, radius, shape, group_map=None,
                                     dtype=F64, outputs=("vmax", "first", "count")):
        """Range-limited merged visibility (vhp_visibility_merge_range_batch): visibility_merge_batch where each
        source only covers the cells in its range, |dx|, |dy| <= radius (shape RANGE_BOX) or
        dx^2 + dy^2 <= radius^2 (RANGE_DISK)."""
        return self._merge_host(self.lib.vhp_visibility_merge_range_batch, (int(radius), int(shape)), occ, src_xy,
                                group_ptr, threshold, group_map, dtype, outputs)

    def visibility_merge_view_batch(self, occ, src_xy, views, group_ptr, threshold, radius, shape, group_map=None,
                                    dtype=F64, outputs=("vmax", "first", "count")):
        """Directional merged visibility (vhp_visibility_merge_view_batch): visibility_merge_range_batch where each
        source only covers the cells in its view.  views: int32 (nsrc, 5), (r, ax, ay, bx, by) per source, the rule of
        visibility_cover_greedy_view_batch (see sensor_views)."""
        vw = np.ascontiguousarray(views, dtype=np.int32).reshape(-1, 5)
        return self._merge_host(self.lib.vhp_visibility_merge_view_batch, (int(radius), int(shape)), occ, src_xy,
                                group_ptr, threshold, group_map, dtype, outputs, views=vw)

    def _merge_host(self, fn, extra, occ, src_xy, group_ptr, threshold, group_map, dtype, outputs, views=None):
        occ = _occ_u8(occ)
        nmaps, ny, nx = occ.shape
        xy = np.ascontiguousarray(src_xy, dtype=np.int32).reshape(-1, 2)
        if views is not None and views.shape[0] != xy.shape[0]:
            raise ValueError(f"views must have one row per source ({xy.shape[0]}), got {views.shape[0]}")
        lead = () if views is None else (_np_ptr(views),)
        gp = np.ascontiguousarray(group_ptr, dtype=np.int64)
        ng = gp.shape[0] - 1
        gm = None if group_map is None else np.ascontiguousarray(group_map, dtype=np.int32)
        kinds = dict(vmax=np.float32 if dtype == F32 else np.float64, first=np.int32, count=np.uint32)
        if set(outputs) - set(kinds):
            raise ValueError(f"outputs are among {tuple(kinds)}")
        r = {k: np.empty((max(ng, 0), ny, nx), kinds[k]) for k in outputs}
        mo = MergeOut(*[_np_ptr(r.get(k)) for k in ("vmax", "first", "count")])
        self._check(fn(self.h, _np_ptr(occ), nmaps, nx, ny, _np_ptr(xy), *lead, _np_ptr(gp), _np_ptr(gm), ng, *extra,
                       float(threshold), dtype, C.byref(mo)))
        return r

    def visibility_merge_batch_dev(self, occ_t, src_xy_t, group_ptr_t, threshold, vmax_t=None, first_t=None,
                                   count_t=None, group_map_t=None):
        """The same on CUDA tensors (asynchronous): occ_t uint8 (nmaps, ny, nx), src_xy_t int32 (nsrc, 2),
        group_ptr_t int64 (ngroups + 1), outputs (ngroups, ny, nx): vmax_t float32/64, first_t int32,
        count_t int32 (read as uint32); any may be None."""
        self._merge_dev(self.lib.vhp_visibility_merge_batch_dev, (), occ_t, src_xy_t, group_ptr_t, threshold, vmax_t,
                        first_t, count_t, group_map_t)

    def visibility_merge_range_batch_dev(self, occ_t, src_xy_t, group_ptr_t, threshold, radius, shape, vmax_t=None,
                                         first_t=None, count_t=None, group_map_t=None):
        """visibility_merge_range_batch on CUDA tensors (asynchronous), arguments as visibility_merge_batch_dev."""
        self._merge_dev(self.lib.vhp_visibility_merge_range_batch_dev, (int(radius), int(shape)), occ_t, src_xy_t,
                        group_ptr_t, threshold, vmax_t, first_t, count_t, group_map_t)

    def visibility_merge_view_batch_dev(self, occ_t, src_xy_t, views_t, group_ptr_t, threshold, radius, shape,
                                        vmax_t=None, first_t=None, count_t=None, group_map_t=None):
        """visibility_merge_view_batch on CUDA tensors (asynchronous), arguments as visibility_merge_batch_dev plus
        views_t int32 (nsrc, 5).  A bad view is reported by the next synchronising call."""
        self._merge_dev(self.lib.vhp_visibility_merge_view_batch_dev, (int(radius), int(shape)), occ_t, src_xy_t,
                        group_ptr_t, threshold, vmax_t, first_t, count_t, group_map_t, views_t=views_t)

    def _merge_dev(self, fn, extra, occ_t, src_xy_t, group_ptr_t, threshold, vmax_t, first_t, count_t, group_map_t,
                   views_t=False):
        nmaps, ny, nx = occ_t.shape
        ng = group_ptr_t.shape[0] - 1
        dtype = F32 if (vmax_t is not None and vmax_t.element_size() == 4) else F64
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        mo = MergeOut(ptr(vmax_t), ptr(first_t), ptr(count_t))
        lead = () if views_t is False else (ptr(views_t),)
        self._check(fn(self.h, occ_t.data_ptr(), nmaps, nx, ny, src_xy_t.data_ptr(), *lead, group_ptr_t.data_ptr(),
                       ptr(group_map_t), ng, src_xy_t.shape[0], *extra, float(threshold), dtype, C.byref(mo)))

    def visibility_cover_greedy_batch(self, occ, cand_xy, group_ptr, k, threshold, radius, shape, group_map=None,
                                      target=None):
        """Greedy sensor placement (vhp_visibility_cover_greedy_batch): per problem q (candidates
        cand_xy[group_ptr[q]:group_ptr[q + 1]] on map group_map[q]) the k candidates, picked one by one, that each add
        the most cells to what the earlier picks cover, within the candidate's range (radius, shape as
        visibility_merge_range_batch) at fp64 value >= threshold.  target: bool (nprob, ny, nx), the cells that count
        (None: all).  Returns pick (int32 (nprob, k), index within the group, -1 after the last pick), gain (uint32
        (nprob, k), cells newly covered), npicked (int32 (nprob,)) and covered (uint32 (nprob, ny, ceil(nx/32)), the
        bits of the union, see unpack_bits)."""
        return self._cover_host(self.lib.vhp_visibility_cover_greedy_batch, CoverOut, occ, cand_xy, group_ptr, k,
                                threshold, radius, shape, group_map, target=target)

    def visibility_cover_greedy_batch_dev(self, occ_t, cand_xy_t, group_ptr_t, k, threshold, radius, shape,
                                          pick_t=None, gain_t=None, npicked_t=None, covered_t=None, group_map_t=None,
                                          target_t=None):
        """The same on CUDA tensors (asynchronous): occ_t uint8 (nmaps, ny, nx), cand_xy_t int32 (nsrc, 2),
        group_ptr_t int64 (nprob + 1), target_t int32 (nprob, ny, ceil(nx/32)) packed bits or None; outputs pick_t,
        gain_t int32 (nprob, k), npicked_t int32 (nprob,), covered_t int32 (nprob, ny, ceil(nx/32)); any may be None."""
        self._cover_dev(self.lib.vhp_visibility_cover_greedy_batch_dev, CoverOut, occ_t, cand_xy_t, group_ptr_t, k,
                        threshold, radius, shape, (pick_t, gain_t, npicked_t, covered_t), group_map_t, target_t)

    def visibility_cover_greedy_weighted_batch(self, occ, cand_xy, group_ptr, k, threshold, radius, shape,
                                               weights=None, group_map=None):
        """Weighted greedy sensor placement (vhp_visibility_cover_greedy_weighted_batch): as
        visibility_cover_greedy_batch, but each round takes the candidate whose newly covered cells have the largest
        summed weight.  weights: uint8 (nprob, ny, nx), the importance of each cell to each problem (None: every cell
        weighs 1).  Returns pick (int32 (nprob, k)), gain (uint64 (nprob, k), summed weight newly covered), npicked
        (int32 (nprob,)) and covered (uint32 (nprob, ny, ceil(nx/32)), the bits of the union, see unpack_bits)."""
        return self._cover_host(self.lib.vhp_visibility_cover_greedy_weighted_batch, CoverWeightedOut, occ, cand_xy,
                                group_ptr, k, threshold, radius, shape, group_map, weights=weights)

    def visibility_cover_greedy_weighted_batch_dev(self, occ_t, cand_xy_t, group_ptr_t, k, threshold, radius, shape,
                                                   pick_t=None, gain_t=None, npicked_t=None, covered_t=None,
                                                   group_map_t=None, weights_t=None):
        """The same on CUDA tensors (asynchronous): occ_t uint8 (nmaps, ny, nx), cand_xy_t int32 (nsrc, 2),
        group_ptr_t int64 (nprob + 1), weights_t uint8 (nprob, ny, nx) or None; outputs pick_t int32 (nprob, k),
        gain_t int64 / uint64 (nprob, k), npicked_t int32 (nprob,), covered_t int32 (nprob, ny, ceil(nx/32)); any may
        be None."""
        self._cover_dev(self.lib.vhp_visibility_cover_greedy_weighted_batch_dev, CoverWeightedOut, occ_t, cand_xy_t,
                        group_ptr_t, k, threshold, radius, shape, (pick_t, gain_t, npicked_t, covered_t), group_map_t,
                        weights_t)

    def visibility_cover_greedy_mfold_batch(self, occ, cand_xy, group_ptr, k, m, threshold, radius, shape,
                                            weights=None, group_map=None):
        """Redundant (m-fold) greedy sensor placement (vhp_visibility_cover_greedy_mfold_batch): as
        visibility_cover_greedy_weighted_batch, but a cell's weight counts until m (1..255) picks cover it, so each
        round takes the candidate, not yet picked, whose cells covered fewer than m times weigh the most.  Returns pick
        (int32 (nprob, k)), gain (uint64 (nprob, k), summed weight the pick adds), npicked (int32 (nprob,)) and count
        (uint8 (nprob, ny, nx), min(m, number of picks covering the cell))."""
        return self._cover_host(self.lib.vhp_visibility_cover_greedy_mfold_batch, CoverMfoldOut, occ, cand_xy,
                                group_ptr, k, threshold, radius, shape, group_map, weights=weights, m=m)

    def visibility_cover_greedy_mfold_batch_dev(self, occ_t, cand_xy_t, group_ptr_t, k, m, threshold, radius, shape,
                                                pick_t=None, gain_t=None, npicked_t=None, count_t=None,
                                                group_map_t=None, weights_t=None):
        """The same on CUDA tensors (asynchronous): occ_t uint8 (nmaps, ny, nx), cand_xy_t int32 (nsrc, 2),
        group_ptr_t int64 (nprob + 1), weights_t uint8 (nprob, ny, nx) or None; outputs pick_t int32 (nprob, k),
        gain_t int64 / uint64 (nprob, k), npicked_t int32 (nprob,), count_t uint8 (nprob, ny, nx); any may be None."""
        self._cover_dev(self.lib.vhp_visibility_cover_greedy_mfold_batch_dev, CoverMfoldOut, occ_t, cand_xy_t,
                        group_ptr_t, k, threshold, radius, shape, (pick_t, gain_t, npicked_t, count_t), group_map_t,
                        weights_t, m=m)

    def visibility_cover_greedy_view_batch(self, occ, cand_xy, views, group_ptr, k, m, threshold, radius, shape,
                                           weights=None, group_map=None):
        """Directional greedy sensor placement (vhp_visibility_cover_greedy_view_batch): as
        visibility_cover_greedy_mfold_batch, with each candidate's coverage narrowed to its view.  views: int32
        (nsrc, 5), (r, ax, ay, bx, by) per candidate: range r (0 <= r <= radius) in the call's shape and the sector
        from a = (ax, ay) to b = (bx, by), in the grid's (x, y) = (column, row); see sensor_views.  Returns pick, gain,
        npicked and count as visibility_cover_greedy_mfold_batch."""
        return self._cover_host(self.lib.vhp_visibility_cover_greedy_view_batch, CoverMfoldOut, occ, cand_xy,
                                group_ptr, k, threshold, radius, shape, group_map, weights=weights, m=m, views=views)

    def visibility_cover_greedy_view_batch_dev(self, occ_t, cand_xy_t, views_t, group_ptr_t, k, m, threshold, radius,
                                               shape, pick_t=None, gain_t=None, npicked_t=None, count_t=None,
                                               group_map_t=None, weights_t=None):
        """The same on CUDA tensors (asynchronous): occ_t uint8 (nmaps, ny, nx), cand_xy_t int32 (nsrc, 2), views_t
        int32 (nsrc, 5), group_ptr_t int64 (nprob + 1), weights_t uint8 (nprob, ny, nx) or None; outputs pick_t int32
        (nprob, k), gain_t int64 / uint64 (nprob, k), npicked_t int32 (nprob,), count_t uint8 (nprob, ny, nx); any may
        be None.  A bad view is reported by the next synchronising call."""
        self._cover_dev(self.lib.vhp_visibility_cover_greedy_view_batch_dev, CoverMfoldOut, occ_t, cand_xy_t,
                        group_ptr_t, k, threshold, radius, shape, (pick_t, gain_t, npicked_t, count_t), group_map_t,
                        weights_t, m=m, views_t=views_t)

    def _cover_host(self, fn, out_type, occ, cand_xy, group_ptr, k, threshold, radius, shape, group_map, target=None,
                    weights=None, m=None, views=None):
        # out_type's fields name the outputs: CoverOut has uint32 gains, the weighted calls' uint64 ones
        occ = _occ_u8(occ)
        nmaps, ny, nx = occ.shape
        xy = np.ascontiguousarray(cand_xy, dtype=np.int32).reshape(-1, 2)
        lead = ()
        if views is not None:
            vw = np.ascontiguousarray(views, dtype=np.int32).reshape(-1, 5)
            if vw.shape[0] != xy.shape[0]:
                raise ValueError(f"views must have one row per candidate ({xy.shape[0]}), got {vw.shape[0]}")
            lead = (_np_ptr(vw),)
        gp = np.ascontiguousarray(group_ptr, dtype=np.int64)
        npb = gp.shape[0] - 1
        n = max(npb, 0)
        gm = None if group_map is None else np.ascontiguousarray(group_map, dtype=np.int32)
        if target is not None:
            extra = pack_bits(np.asarray(target, bool).reshape(n, ny, nx))
        else:
            extra = _cover_weights(weights, (n, ny, nx))
        k = int(k)
        kinds = dict(pick=((n, max(k, 0)), np.int32),
                     gain=((n, max(k, 0)), np.uint32 if out_type is CoverOut else np.uint64),
                     npicked=((n,), np.int32), covered=((n, ny, (nx + 31) // 32), np.uint32),
                     count=((n, ny, nx), np.uint8))
        names = [name for name, _ in out_type._fields_]
        r = {name: np.empty(*kinds[name]) for name in names}
        co = out_type(*[_np_ptr(r[name]) for name in names])
        tail = () if m is None else (int(m),)
        self._check(fn(self.h, _np_ptr(occ), nmaps, nx, ny, _np_ptr(xy), *lead, _np_ptr(gp), _np_ptr(gm), npb, k,
                       int(radius), int(shape), float(threshold), _np_ptr(extra), *tail, C.byref(co)))
        return r

    def _cover_dev(self, fn, out_type, occ_t, cand_xy_t, group_ptr_t, k, threshold, radius, shape, outs, group_map_t,
                   extra_t, m=None, views_t=False):
        nmaps, ny, nx = occ_t.shape
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        co = out_type(*[ptr(t) for t in outs])
        lead = () if views_t is False else (ptr(views_t),)
        tail = () if m is None else (int(m),)
        self._check(fn(self.h, occ_t.data_ptr(), nmaps, nx, ny, cand_xy_t.data_ptr(), *lead, group_ptr_t.data_ptr(),
                       ptr(group_map_t), group_ptr_t.shape[0] - 1, cand_xy_t.shape[0], int(k), int(radius),
                       int(shape), float(threshold), ptr(extra_t), *tail, C.byref(co)))

    def visibility_variant_batch(self, occ, src_xy, model, alpha=1.0, fac=1.0, light_strength=1.0,
                                 cutoff=0.001, src_map=None, dtype=F64):
        """Opt-in sweep variants (vhp_visibility_variant_batch): VARIANT_MATLAB =
        getAccessibilityMap.m with decay alpha / curve factor fac, VARIANT_QUEUE = the
        early-terminating computeVisibilityUsingQueue rule."""
        var = SweepVariant(int(model), float(alpha), float(fac), float(light_strength), float(cutoff))

        def fn(h, occ_p, nmaps, nx, ny, xy_p, mp_p, n, dt, out_p):
            return self.lib.vhp_visibility_variant_batch(h, occ_p, nmaps, nx, ny, xy_p, mp_p, n, C.byref(var), dt, out_p)
        return self._batch_host(fn, occ, src_xy, src_map, dtype, None)

    def raycast_batch(self, occ, src_xy, src_map=None, dtype=F64, out=None):
        return self._batch_host(self.lib.vhp_raycast_batch, occ, src_xy, src_map, dtype, out)

    def planner_batch(self, occ, start_end, prob_map=None, threshold=0.5, max_iter=100,
                      dtype=F64, fields=True, ls_cap=None):
        """solve() + reconstructPath() for every problem.  Returns a dict of numpy
        arrays (status, nb_sources, light_sources, path_len, path_n, path[, vg,
        came, vis]).  ls_cap: entries per problem of light_sources and path (default
        max_iter + 2, the least the library accepts)."""
        occ = _occ_u8(occ)
        nmaps, ny, nx = occ.shape
        se = np.ascontiguousarray(start_end, dtype=np.int32).reshape(-1, 4)
        n = se.shape[0]
        mp = None if prob_map is None else np.ascontiguousarray(prob_map, dtype=np.int32)
        cap = int(max_iter) + 2 if ls_cap is None else int(ls_cap)
        ft = np.float32 if dtype == F32 else np.float64
        r = dict(status=np.zeros(n, np.int32), nb_sources=np.zeros(n, np.int32),
                 light_sources=np.zeros((n, max(cap, 0), 2), np.int32), path_len=np.zeros(n),
                 path_n=np.zeros(n, np.int32), path=np.zeros((n, max(cap, 0), 2), np.int32))
        if fields:
            r.update(vg=np.zeros((n, ny, nx), ft), came=np.zeros((n, ny, nx), np.int32),
                     vis=np.zeros((n, ny, nx), ft))
        po = PlannerOut(*[_np_ptr(r.get(k)) for k in
                          ("status", "nb_sources", "light_sources", "path_len", "path_n",
                           "path", "vg", "came", "vis")])
        self._check(self.lib.vhp_planner_batch(self.h, _np_ptr(occ), nmaps, nx, ny,
                                               _np_ptr(se), _np_ptr(mp), n, float(threshold),
                                               int(max_iter), cap, dtype, C.byref(po)))
        return r

    PLANNER_OUTPUTS = ("status", "nb_sources", "light_sources", "path_len", "path_n", "path", "vg", "came", "vis")

    def planner_batch_dev(self, occ_t, start_end_t, prob_map_t=None, threshold=0.5, max_iter=100, ls_cap=None,
                          dtype=F64, **outputs):
        """planner_batch on CUDA tensors (asynchronous, returns nothing): occ_t uint8 (nmaps, ny, nx),
        start_end_t int32 (nprob, 4), prob_map_t int32 (nprob,) or None.  Outputs by keyword, each a
        contiguous CUDA tensor or omitted: status, nb_sources, path_n int32 (nprob,), path_len float64
        (nprob,), light_sources, path int32 (nprob, ls_cap, 2), came int32 (nprob, ny, nx), vg, vis (nprob,
        ny, nx) of dtype.  With no output at all the library gets a NULL output struct."""
        unknown = set(outputs) - set(self.PLANNER_OUTPUTS)
        if unknown:
            raise ValueError(f"unknown planner outputs {sorted(unknown)}; they are among {self.PLANNER_OUTPUTS}")
        for k in ("vg", "vis"):
            t = outputs.get(k)
            if t is not None and t.element_size() != (4 if dtype == F32 else 8):
                raise ValueError(f"{k} must be of the dtype of the call")
        nmaps, ny, nx = occ_t.shape
        cap = int(max_iter) + 2 if ls_cap is None else int(ls_cap)
        po = None
        if any(t is not None for t in outputs.values()):
            po = C.byref(PlannerOut(*[None if outputs.get(k) is None else outputs[k].data_ptr()
                                      for k in self.PLANNER_OUTPUTS]))
        self._check(self.lib.vhp_planner_batch_dev(
            self.h, occ_t.data_ptr(), nmaps, nx, ny, start_end_t.data_ptr(),
            None if prob_map_t is None else prob_map_t.data_ptr(), start_end_t.shape[0], float(threshold),
            int(max_iter), cap, dtype, po))

    # ---- device (torch) entry points ----------------------------------------
    def visibility_batch_dev(self, occ_t, src_xy_t, out_t, src_map_t=None):
        """occ_t uint8 (nmaps, ny, nx), src_xy_t int32 (n, 2), out_t float32/64
        (n, ny, nx); all CUDA tensors, contiguous.  Asynchronous."""
        nmaps, ny, nx = occ_t.shape
        dtype = F32 if out_t.element_size() == 4 else F64
        self._check(self.lib.vhp_visibility_batch_dev(
            self.h, occ_t.data_ptr(), nmaps, nx, ny, src_xy_t.data_ptr(),
            None if src_map_t is None else src_map_t.data_ptr(), src_xy_t.shape[0], dtype,
            out_t.data_ptr()))

    def visibility_window_batch_dev(self, occ_t, src_xy_t, radius, out_t, src_map_t=None):
        """The same on CUDA tensors (asynchronous): occ_t uint8 (nmaps, ny, nx), src_xy_t int32 (n, 2),
        out_t float32/64 (n, 2R+1, 2R+1), contiguous."""
        nmaps, ny, nx = occ_t.shape
        dtype = F32 if out_t.element_size() == 4 else F64
        self._check(self.lib.vhp_visibility_window_batch_dev(
            self.h, occ_t.data_ptr(), nmaps, nx, ny, src_xy_t.data_ptr(),
            None if src_map_t is None else src_map_t.data_ptr(), src_xy_t.shape[0], int(radius), dtype,
            out_t.data_ptr()))

    def raycast_batch_dev(self, occ_t, src_xy_t, out_t, src_map_t=None):
        nmaps, ny, nx = occ_t.shape
        dtype = F32 if out_t.element_size() == 4 else F64
        self._check(self.lib.vhp_raycast_batch_dev(
            self.h, occ_t.data_ptr(), nmaps, nx, ny, src_xy_t.data_ptr(),
            None if src_map_t is None else src_map_t.data_ptr(), src_xy_t.shape[0], dtype,
            out_t.data_ptr()))

    def generate_environments_dev(self, occ_t, nb_of_obstacles, min_w, max_w, min_h, max_h, seed,
                                  first_map=0):
        """Fill occ_t (uint8 CUDA tensor (nmaps, ny, nx)) with random-rectangle environments
        first_map .. first_map + nmaps - 1 of the family `seed` (vhp_environment_generate_batch_dev)."""
        nmaps, ny, nx = occ_t.shape
        cfg = Config()
        self.lib.vhp_config_default(C.byref(cfg))
        cfg.ncols, cfg.nrows, cfg.nb_of_obstacles = nx, ny, int(nb_of_obstacles)
        cfg.min_width, cfg.max_width, cfg.min_height, cfg.max_height = int(min_w), int(max_w), int(min_h), int(max_h)
        self._check(self.lib.vhp_environment_generate_batch_dev(self.h, C.byref(cfg), int(seed),
                                                                int(first_map), nmaps, occ_t.data_ptr()))

    def prepare_maps_dev(self, occ_t):
        nmaps, ny, nx = occ_t.shape
        self._check(self.lib.vhp_prepare_maps_dev(self.h, occ_t.data_ptr(), nmaps, nx, ny))


def runs_to_bits(row_count, pair_ptr, trans, nx):
    """Row runs -> uint32 bit maps (npairs, ny, ceil(nx/32)) (vhp_runs_to_bits)."""
    lib = load_library()
    n, ny = row_count.shape
    out = np.empty((n, ny, (nx + 31) // 32), np.uint32)
    tr = np.ascontiguousarray(trans, dtype=np.uint16)
    if tr.size == 0:
        tr = np.zeros(1, np.uint16)
    st = lib.vhp_runs_to_bits(_np_ptr(np.ascontiguousarray(row_count)), _np_ptr(np.ascontiguousarray(pair_ptr)),
                              _np_ptr(tr), n, nx, ny, _np_ptr(out))
    if st != 0:
        raise VhpError(st, lib.vhp_last_error(None).decode())
    return out


def unpack_bits(bits, nx):
    """uint32 (..., ceil(nx/32)) bit-packed rows -> bool (..., nx)."""
    b = np.ascontiguousarray(bits).view(np.uint8)
    return np.unpackbits(b, axis=-1, bitorder="little")[..., :nx].astype(bool)


def pack_bits(cells):
    """bool (..., nx) -> uint32 (..., ceil(nx/32)) bit-packed rows (bit x & 31 of word x >> 5), the inverse of
    unpack_bits."""
    cells = np.asarray(cells, bool)
    nx = cells.shape[-1]
    pad = np.zeros(cells.shape[:-1] + (32 * ((nx + 31) // 32),), bool)
    pad[..., :nx] = cells
    return np.ascontiguousarray(np.packbits(pad, axis=-1, bitorder="little")).view("<u4")


def sensor_views(heading_deg, fov_deg, radius, scale=32767):
    """Views for visibility_cover_greedy_view_batch and visibility_merge_view_batch: int32 (n, 5) rows (r, ax, ay, bx, by) from headings and fields of
    view in degrees (scalars or arrays, broadcast together).  Angles are measured from +x (the column) towards +y (the
    row).  a = round(scale * dir(heading - fov / 2)) and b = round(scale * dir(heading + fov / 2)); fov >= 360 gives
    a == b = round(scale * dir(heading)), every direction.  The library sees only these integer vectors: they, not the
    angles, define the view, so a sector edge is the rounded direction (at scale 32767 within about 2e-3 degrees).
    Raises ValueError when fov <= 0, scale is outside [1, 32767], or fov < 360 but the rounded a and b point the same
    way, which the library would read as every direction."""
    h, f, r = np.broadcast_arrays(np.asarray(heading_deg, np.float64), np.asarray(fov_deg, np.float64),
                                  np.asarray(radius, np.int64))
    h, f, r = h.reshape(-1), f.reshape(-1), r.reshape(-1)
    if not 1 <= int(scale) <= 32767:
        raise ValueError(f"scale must be in [1, 32767], got {scale}")
    if (f <= 0).any():
        raise ValueError("fov must be positive")
    full = f >= 360
    half = np.where(full, 0.0, f / 2)
    ta, tb = np.radians(h - half), np.radians(h + half)
    a = np.rint(int(scale) * np.stack([np.cos(ta), np.sin(ta)], 1)).astype(np.int64)
    b = np.rint(int(scale) * np.stack([np.cos(tb), np.sin(tb)], 1)).astype(np.int64)
    cross = a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]
    dot = a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]
    same = (cross == 0) & (dot > 0) & ~full
    if same.any():
        i = int(np.flatnonzero(same)[0])
        raise ValueError(f"fov {f[i]} at heading {h[i]}: the rounded sector edges point the same way "
                         f"(a = {tuple(a[i])}, b = {tuple(b[i])}); use a larger fov or scale")
    return np.ascontiguousarray(np.concatenate([r[:, None], a, b], 1).astype(np.int32))


def torch_context(device: int, stream) -> Context:
    """Context that enqueues on the given torch.cuda.Stream (time it with events
    recorded on that stream)."""
    return Context(device, C.c_void_p(stream.cuda_stream))
