"""ctypes binding of libmpb200.so (include/mpb200.h).

There is deliberately no fallback: if the CUDA library is missing or no B200 is present the
first compute call raises.  The oracle under /oracle is test infrastructure and is never
imported from here.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libmpb200.so")

c_i64 = ctypes.c_int64
c_i32 = ctypes.c_int32
c_dbl = ctypes.c_double
c_vp = ctypes.c_void_p
P = ctypes.POINTER


class MPB200Error(RuntimeError):
    """Raised for any non-zero return of the C ABI (mirrors the reference's `error(...)`)."""


class ObstaclesDesc(ctypes.Structure):
    _fields_ = [
        ("n_gates", c_i32), ("gate_parent", c_vp), ("gate_aabb", c_vp),
        ("n_shapes", c_i32), ("shape_kind", c_vp), ("shape_gate", c_vp), ("shape_off", c_vp),
        ("data", c_vp), ("flags", c_i32),
    ]


class SpaceDesc(ctypes.Structure):
    _fields_ = [
        ("n", c_i32), ("lo", c_vp), ("hi", c_vp), ("s2w_kind", c_i32), ("dw", c_i32),
        ("inds", c_vp), ("C", c_vp),
    ]


class McProblem(ctypes.Structure):
    _fields_ = [("T", c_i32), ("nz", c_i32), ("q", c_i32), ("dw", c_i32), ("F", c_vp), ("G", c_vp), ("Wz", c_vp),
                ("wbar", c_vp), ("K", c_i32), ("alpha", c_vp), ("mu", c_vp), ("swept", c_i32)]


class McResult(ctypes.Structure):
    _fields_ = [("s1", c_dbl), ("s2", c_dbl), ("s0", c_dbl), ("n", c_i64), ("hits", c_i64)]


class GmtDesc(ctypes.Structure):
    _fields_ = [("fwd", c_vp), ("bwd", c_vp), ("goal_bits", c_vp), ("init", c_i64), ("width", c_dbl),
                ("checkpts", c_i32), ("space", P(SpaceDesc))]


class GmtResult(ctypes.Structure):
    _fields_ = [("solved", c_i32), ("grid_blocks", c_i32), ("goal", c_i64), ("cost", c_dbl), ("iterations", c_i64),
                ("expansions", c_i64), ("checks", c_i64), ("checks_in_bounds", c_i64), ("path_len", c_i64)]


class GmtEdges(ctypes.Structure):
    _fields_ = [("kind", c_i32), ("obstacles", c_vp), ("lq", c_vp), ("r", c_dbl), ("car_kind", c_i32),
                ("turning_radius", c_dbl), ("speed", c_dbl)]


GMT_EDGES_STRAIGHT, GMT_EDGES_LQ, GMT_EDGES_CAR = 0, 1, 2  # mpb200_gmt_edges.kind


# every symbol include/mpb200.h declares: name -> (restype, argtypes)
OP_TABLE, OP_POINTS, OP_EDGES, OP_OTHER, OP_PLAN, OP_PATH = 0, 1, 2, 3, 4, 5  # mpb200_last_ms_of operation kinds

SIGNATURES = {
    "mpb200_init": (ctypes.c_int, [ctypes.c_int]),
    "mpb200_shutdown": (None, []),
    "mpb200_last_error": (ctypes.c_char_p, []),
    "mpb200_version": (ctypes.c_int, []),
    "mpb200_set_stream": (ctypes.c_int, [c_vp]),
    "mpb200_synchronize": (ctypes.c_int, []),
    "mpb200_host_alloc": (ctypes.c_int, [ctypes.c_uint64, P(c_vp)]),
    "mpb200_host_free": (ctypes.c_int, [c_vp]),
    "mpb200_launch_count": (c_i64, []),
    "mpb200_release_cached": (ctypes.c_int, []),
    "mpb200_last_ms": (c_dbl, [ctypes.c_int]),
    "mpb200_last_ms_of": (c_dbl, [ctypes.c_int, ctypes.c_int]),
    "mpb200_samples_create": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, P(c_vp)]),
    "mpb200_sample_free": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.c_uint64, ctypes.c_int32, c_vp, c_vp, c_vp]),
    "mpb200_samples_destroy": (ctypes.c_int, [c_vp]),
    "mpb200_samples_set_query_range": (ctypes.c_int, [c_vp, c_i64, c_i64]),
    "mpb200_inball_build": (ctypes.c_int, [c_vp, c_dbl, P(c_vp), P(c_i64)]),
    "mpb200_table_fetch": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp]),
    "mpb200_inball_build_checked": (ctypes.c_int, [c_vp, c_dbl, c_vp, P(SpaceDesc), P(c_vp), P(c_i64), P(c_i64)]),
    "mpb200_table_fetch_edge_bits": (ctypes.c_int, [c_vp, c_vp]),
    "mpb200_table_nnz": (ctypes.c_int, [c_vp, P(c_i64), P(c_i64)]),
    "mpb200_table_device_view": (ctypes.c_int, [c_vp, P(c_vp), P(c_vp), P(c_vp), P(c_vp)]),
    "mpb200_table_destroy": (ctypes.c_int, [c_vp]),
    "mpb200_obstacles2d_create": (ctypes.c_int, [P(ObstaclesDesc), P(c_vp)]),
    "mpb200_boxes_create": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int, ctypes.c_int, P(c_vp)]),
    "mpb200_obstacles_destroy": (ctypes.c_int, [c_vp]),
    "mpb200_points_free": (ctypes.c_int, [c_vp, c_vp, P(SpaceDesc), c_vp]),
    "mpb200_edges_free": (ctypes.c_int, [c_vp, c_vp, c_vp, P(SpaceDesc), c_vp, P(c_i64)]),
    "mpb200_states_free": (ctypes.c_int, [c_vp, c_i64, ctypes.c_int, c_vp, P(SpaceDesc), c_vp]),
    "mpb200_segments_free": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.c_int, c_vp, P(SpaceDesc), c_vp]),
    "mpb200_lq_create": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, ctypes.c_int, ctypes.c_int, P(c_vp)]),
    "mpb200_lq_destroy": (ctypes.c_int, [c_vp]),
    "mpb200_lq_inball_build": (ctypes.c_int, [c_vp, c_vp, c_dbl, P(c_vp), P(c_vp), P(c_i64), P(c_i64)]),
    "mpb200_lq_steer": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, c_dbl, c_vp, c_vp]),
    "mpb200_lq_edges_free": (ctypes.c_int, [c_vp, c_vp, c_vp, c_dbl, c_vp, P(SpaceDesc), c_vp, P(c_i64)]),
    "mpb200_mc_collision_probability": (ctypes.c_int, [P(McProblem), c_vp, ctypes.c_uint64, c_i64, c_i64, P(McResult),
                                                       c_vp, c_vp]),
    "mpb200_table_knn": (ctypes.c_int, [c_vp, ctypes.c_int, P(c_vp), P(c_i64), P(c_i64)]),
    "mpb200_table_short_columns": (ctypes.c_int, [c_vp, ctypes.c_int, P(c_i64)]),
    "mpb200_table_union_transpose": (ctypes.c_int, [c_vp, c_vp, P(c_vp), P(c_i64)]),
    "mpb200_close_points": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i64, ctypes.c_int, c_dbl, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mpb200_xchg_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, c_i64, c_i64, P(c_vp), c_vp]),
    "mpb200_xchg_connect": (ctypes.c_int, [c_vp, c_vp]),
    "mpb200_xchg_attach": (ctypes.c_int, [c_vp, c_vp]),
    "mpb200_xchg_push": (ctypes.c_int, [c_vp, c_vp]),
    "mpb200_xchg_view": (ctypes.c_int, [c_vp, P(c_vp), P(c_i64), P(c_i64), P(c_i64), P(c_i64)]),
    "mpb200_xchg_destroy": (ctypes.c_int, [c_vp]),
    "mpb200_table_write_floor": (ctypes.c_int, [c_vp, P(c_dbl)]),
    "mpb200_pipe_peak": (ctypes.c_int, [ctypes.c_int, P(c_dbl)]),
    "mpb200_car_inball_build": (ctypes.c_int, [c_vp, ctypes.c_int32, c_dbl, c_dbl, c_dbl, P(c_vp), P(c_vp), P(c_i64), P(c_i64)]),
    "mpb200_car_last_candidates": (ctypes.c_int, [c_vp, P(c_i64)]),
    "mpb200_car_steer": (ctypes.c_int, [ctypes.c_int32, c_dbl, c_dbl, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "mpb200_car_edges_free": (ctypes.c_int, [c_vp, c_vp, ctypes.c_int32, c_dbl, c_dbl, c_vp, P(SpaceDesc), c_vp, P(c_i64)]),
    "mpb200_car_motions_free": (ctypes.c_int, [ctypes.c_int32, c_dbl, c_dbl, c_vp, c_vp, c_i64, c_vp, P(SpaceDesc), c_vp, P(c_i64)]),
    "mpb200_lq_motions_free": (ctypes.c_int, [c_vp, c_dbl, c_vp, c_vp, c_i64, c_vp, P(SpaceDesc), c_vp, P(c_i64)]),
    "mpb200_gmt_plan": (ctypes.c_int, [c_vp, P(GmtDesc), P(GmtResult), c_vp, c_i64, c_vp, c_vp]),
    "mpb200_gmt_plan_lazy": (ctypes.c_int, [c_vp, P(GmtDesc), P(GmtEdges), P(GmtResult), P(c_i64), c_vp, c_i64, c_vp,
                                            c_vp]),
    "mpb200_gmt_plan_batch": (ctypes.c_int, [c_vp, P(GmtDesc), c_i64, P(GmtEdges), P(GmtResult), c_vp, c_vp, c_i64,
                                             c_vp, c_vp]),
    "mpb200_shortcut_paths": (ctypes.c_int, [c_vp, c_vp, c_i64, ctypes.c_int, c_vp, P(SpaceDesc), c_i32, c_vp, c_i64,
                                             c_vp, c_vp, c_vp, c_vp]),
}

_lib = None
_initialised = False


def load():
    """dlopen the library and declare every signature (no GPU needed for this)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MPB200Error(
                "libmpb200.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `python motionplanning.jl_b200/build.py`. There is no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        msg = load().mpb200_last_error()
        raise MPB200Error("libmpb200 error %d: %s" % (rc, msg.decode() if msg else "?"))


def init(device=None):
    """Bind this process to one GPU (LOCAL_RANK by default) -- one process per GPU."""
    global _initialised
    lib = load()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    check(lib.mpb200_init(int(device)))
    _initialised = True
    return lib


def lib():
    """The initialised library; raises if there is no usable B200."""
    if not _initialised:
        return init()
    return _lib


def ptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(c_vp)


class _PinnedBlock:
    """One cudaMallocHost allocation, freed when the last numpy array over it is collected (the arrays
    keep this object as their base), so a result array can never outlive its memory."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        p = c_vp()
        check(lib().mpb200_host_alloc(self.nbytes, ctypes.byref(p)))
        self.ptr = p.value
        self.__array_interface__ = {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 3}

    def __del__(self):
        try:
            if self.ptr and _lib is not None:
                _lib.mpb200_host_free(c_vp(self.ptr))
        except Exception:
            pass
        self.ptr = None


class PinnedPool:
    """Pinned host result arrays (D2H at PCIe speed).

    Default: every array() call returns a freshly allocated, OWNING array -- it stays valid for as long as
    the caller keeps it, whatever happens to the sample set, the pool or later precomputes (ImmutableNNC is
    immutable).  reuse=True is the explicit opt-in of the benchmark loop: arrays with the same key alias ONE
    buffer that the next request overwrites in place; the memory itself still lives until the last array
    over it is dropped (reference counted), so even then nothing dangles."""

    def __init__(self, reuse=False):
        self.reuse = bool(reuse)
        self._bufs = {}

    def array(self, key, n, dtype):
        dtype = np.dtype(dtype)
        nbytes = max(int(n) * dtype.itemsize, 8)
        if not self.reuse:
            if nbytes < (1 << 20):   # small results: a pageable array (pinning costs more than it saves)
                return np.empty(int(n), dtype=dtype)
            block = _PinnedBlock(nbytes)
        else:
            block = self._bufs.get(key)
            if block is None or block.nbytes < nbytes:
                block = _PinnedBlock(nbytes + nbytes // 8)   # the outgrown block is dropped, not freed under its views
                self._bufs[key] = block
        return np.asarray(block)[:int(n) * dtype.itemsize].view(dtype)

    def release(self):
        self._bufs.clear()
