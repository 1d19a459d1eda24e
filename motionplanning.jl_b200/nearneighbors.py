"""Near-neighbour sample sets served from GPU-built tables.

Mirror of src/nearneighbors.jl: SampleSet / MetricNN (:62-74), ImmutableNNC (:23-28),
filter_neighborhood (:104-107), the cached inball!/inballF!/inballB! dispatch (:120-136,200-203)
and viewcol (src/utilities/utils.jl:76-82).  Where the reference fills a MutableNNC lazily, one
query at a time through a KD-tree (geometric.jl:14; nearneighbors.jl:179-183), this back-end
builds the whole ImmutableNNC.D matrix in one GPU pass (mpb200_inball_build) and serves columns
with viewcol -- the seam the reference already has at nearneighbors.jl:128.

Indices are 1-based Int64 exactly as in Julia's SparseMatrixCSC, so the arrays can be handed to
`SparseMatrixCSC(N, N, colptr, rowval, nzval)` unchanged.
"""
import ctypes

import numpy as np

from . import _lib
from .statespaces import Euclidean


class SparseMatrixCSC:
    """Field-for-field Julia SparseMatrixCSC{Float64,Int64} (1-based colptr/rowval)."""

    def __init__(self, m, n, colptr, rowval, nzval):
        self.m, self.n = int(m), int(n)
        self.colptr, self.rowval, self.nzval = colptr, rowval, nzval

    @property
    def nnz(self):
        return int(self.colptr[-1] - 1)


class SparseVectorView:
    """utils.jl:63-75"""

    def __init__(self, n, nzind, nzval):
        self.n, self.nzind, self.nzval = n, nzind, nzval

    def __len__(self):
        return self.n


def nonzeroinds(x):
    return x.nzind


def nonzeros(x):
    return x.nzval


def viewcol(x, j):
    """utils.jl:76-82 (j is 1-based)"""
    if not 1 <= j <= x.n:
        raise IndexError("BoundsError")
    r1 = int(x.colptr[j - 1]) - 1
    r2 = int(x.colptr[j]) - 1
    return SparseVectorView(x.m, x.rowval[r1:r2], x.nzval[r1:r2])


def filter_neighborhood(n, f):
    """nearneighbors.jl:104-107; f is a boolean mask indexed by 0-based sample position."""
    inds, ds = n.nzind, n.nzval
    keep = f[inds - 1]
    return SparseVectorView(n.n, inds[keep], ds[keep])


class ImmutableNNC:
    """nearneighbors.jl:23-28 -- a fully precomputed neighbour table; `r` is informational
    (the reference never re-validates it, SURVEY quirk Q7)."""

    def __init__(self, D, r):
        self.D = D
        self.r = r


def saveNN(path, cache, edge_chunks=None, point_chunks=None):
    """On-disk form of a precomputed neighbour table and its validity sidecars (SURVEY 8(f).2).  The reference
    exports the names only (`# export saveNN, loadNN!`, nearneighbors.jl:8; the "Serialization" section :114-116
    is empty); the format here is the SparseMatrixCSC fields as they cross the C ABI (1-based Int64 colptr /
    rowval, Float64 nzval) plus the BitVector chunks of the edge and point validity tables, in one .npz."""
    D = cache.D
    arrays = dict(m=np.int64(D.m), n=np.int64(D.n), r=np.float64(cache.r), colptr=np.asarray(D.colptr, dtype=np.int64),
                  rowval=np.asarray(D.rowval, dtype=np.int64), nzval=np.asarray(D.nzval, dtype=np.float64))
    if edge_chunks is not None:
        arrays["edge_chunks"] = np.asarray(edge_chunks, dtype=np.uint64)
    if point_chunks is not None:
        arrays["point_chunks"] = np.asarray(point_chunks, dtype=np.uint64)
    np.savez(path, **arrays)


def loadNN(path, NN=None):
    """Inverse of saveNN -> (ImmutableNNC, edge_chunks or None, point_chunks or None); installs the cache into
    `NN` (a MetricNN) when given, like loadNN! would."""
    with np.load(path) as z:
        D = SparseMatrixCSC(int(z["m"]), int(z["n"]), z["colptr"], z["rowval"], z["nzval"])
        cache = ImmutableNNC(D, float(z["r"]))
        edge = z["edge_chunks"] if "edge_chunks" in z.files else None
        pts = z["point_chunks"] if "point_chunks" in z.files else None
    if D.colptr[0] != 1 or len(D.colptr) != D.n + 1 or D.nnz != len(D.rowval) or D.nnz != len(D.nzval):
        raise ValueError("%s does not hold a consistent CSC table" % path)
    if edge is not None and len(edge) != (D.nnz + 63) // 64:
        raise ValueError("edge validity sidecar does not match the table")
    if NN is not None:
        if len(NN) != D.m:
            raise ValueError("table is for %d samples, the sample set has %d" % (D.m, len(NN)))
        NN.cache = cache
    return cache, edge, pts


class DeviceTable:
    """Owner of a device-resident CSC table handle (mpb200_table)."""

    def __init__(self, name="nn"):
        self.h = _lib.c_vp()
        self.nnz = 0
        self.ncols = 0
        self.name = name  # role of the table ("nn", "F", "B"): keys the reusable pinned result buffers

    def close(self):
        if self.h:
            _lib.load().mpb200_table_destroy(self.h)
            self.h = _lib.c_vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SampleSet:
    """nearneighbors.jl:14 -- common part of MetricNN / QuasiMetricNN: the sample matrix on the
    host (N x d, one state per row == Julia's d x N column-major) and its device copy."""

    def __init__(self, V, dist, init):
        self.V = np.ascontiguousarray(V, dtype=np.float64)
        if self.V.ndim != 2:
            raise ValueError("V must be an N x d array (one state per row)")
        self.dist = dist
        self.init = np.asarray(init, dtype=np.float64)
        self._handle = None
        self.q0, self.q1 = 0, self.V.shape[0]
        self.pool = _lib.PinnedPool()

    def __len__(self):
        return self.V.shape[0]

    def __getitem__(self, i):
        """nearneighbors.jl:111 -- 1-based; NN[0] is the init state"""
        return self.V[i - 1] if i > 0 else self.init

    def handle(self):
        if self._handle is None:
            lib = _lib.lib()
            h = _lib.c_vp()
            _lib.check(lib.mpb200_samples_create(_lib.ptr(self.V), self.V.shape[0], self.V.shape[1], ctypes.byref(h)))
            self._handle = h
            if (self.q0, self.q1) != (0, self.V.shape[0]):
                _lib.check(lib.mpb200_samples_set_query_range(h, self.q0, self.q1))
        return self._handle

    @classmethod
    def sample_free(cls, CC, SS, N, seed=0, init=None, order="candidate", **kw):
        """Sample set of N free states generated, tested and compacted on the device (mpb200_sample_free; the
        bulk of sample_free!, sampling.jl:23-37): the samples never cross PCIe on their way in, the host copy
        `V` is fetched once for the planner.  `candidates` = states drawn to find them.  Deterministic in
        (CC, SS, N, seed); the candidate stream is specified in oracle/sample.c.  order="morton" numbers the
        samples along a Z-order curve instead of in draw order (same set; the table kernels run ~12% faster)."""
        N = int(N)
        V = np.empty((N, SS.dim), dtype=np.float64)
        d = SS.desc()
        h = _lib.c_vp()
        used = _lib.c_i64(0)
        _lib.check(_lib.lib().mpb200_sample_free(CC.handle(), ctypes.byref(d), N, int(seed) & (2**64 - 1),
                                                 {"candidate": 0, "morton": 1}[order], ctypes.byref(h),
                                                 _lib.ptr(V), ctypes.byref(used)))
        obj = cls(V, init=(init if init is not None else (V[0] if N else np.zeros(SS.dim))), **kw)
        obj._handle = h
        obj.candidates = used.value
        return obj

    def set_query_range(self, q0, q1):
        """Multi-GPU shard: this process owns query columns [q0, q1) (0-based)."""
        self.q0, self.q1 = int(q0), int(q1)
        if self._handle is not None:
            _lib.check(_lib.lib().mpb200_samples_set_query_range(self._handle, self.q0, self.q1))

    def close(self):
        if self._handle is not None:
            _lib.load().mpb200_samples_destroy(self._handle)
            self._handle = None
        self.pool.release()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- batched validity over this sample set --------------------------------------------
    def points_free(self, CC, SS, fetch=True):
        """F[i] = is_free_state(V[i], CC, SS) for the owned samples [q0, q1) -- all of them unless a
        query range is set -- (fmt.jl:31-36) as BitVector chunks."""
        n = self.q1 - self.q0
        d = SS.desc()
        bits = self.pool.array("point_bits", (n + 63) // 64, np.uint64) if fetch else None
        _lib.check(_lib.lib().mpb200_points_free(self.handle(), CC.handle(), ctypes.byref(d), _lib.ptr(bits)))
        return bits

    def edges_free(self, table, CC, SS, fetch=True, count=True):
        """Validity bit per stored entry (row y -> column x) of `table`; returns (chunks, checks).
        fetch=False, count=False only enqueues the work (bits stay on the device, no wait)."""
        d = SS.desc()
        bits = self.pool.array(("edge_bits", table.name), (table.nnz + 63) // 64, np.uint64) if fetch else None
        if not fetch and not count:
            _lib.check(_lib.lib().mpb200_edges_free(self.handle(), table.h, CC.handle(), ctypes.byref(d), None, None))
            return None, None
        checks = _lib.c_i64(0)
        _lib.check(_lib.lib().mpb200_edges_free(self.handle(), table.h, CC.handle(), ctypes.byref(d), _lib.ptr(bits),
                                                ctypes.byref(checks)))
        CC.count += checks.value
        return bits, checks.value

    def fetch_table(self, table, key="nn"):
        """Copy a device table into (pinned, reused) host arrays -> SparseMatrixCSC over the shard."""
        colptr = self.pool.array((key, "colptr"), table.ncols + 1, np.int64)
        rowval = self.pool.array((key, "rowval"), table.nnz, np.int64)
        nzval = self.pool.array((key, "nzval"), table.nnz, np.float64)
        _lib.check(_lib.lib().mpb200_table_fetch(table.h, _lib.ptr(colptr), _lib.ptr(rowval), _lib.ptr(nzval)))
        return SparseMatrixCSC(len(self), table.ncols, colptr, rowval, nzval)


def _is_car(dist):
    from .simplecars import is_car_metric
    return is_car_metric(dist)


def _car_edges_free(NN, table, CC, SS, fetch=True):
    """validity per stored entry (row y -> column x) of a car-space table: the motion V[y] -> V[x] (fmt.jl:75)"""
    m = NN.dist.m
    d = SS.desc()
    bits = NN.pool.array(("car_edge_bits", table.name), (table.nnz + 63) // 64, np.uint64) if fetch else None
    checks = _lib.c_i64(0)
    _lib.check(_lib.lib().mpb200_car_edges_free(NN.handle(), table.h, m.kind, m.r, m.s, CC.handle(), ctypes.byref(d),
                                                _lib.ptr(bits), ctypes.byref(checks)))
    CC.count += checks.value
    return bits, checks.value


def _knn_radius_guess(V, k):
    """radius of the ball expected to hold ~1.6 k samples of a uniform cloud filling the samples' bounding box"""
    import math
    N, d = V.shape
    ext = np.maximum(V.max(axis=0) - V.min(axis=0), 1e-300)
    zeta = math.pi ** (d / 2) / math.gamma(d / 2 + 1)
    # in 2-D / 3-D the columns that decide are the ones in the corners of the box, which see 1/2^d of a ball
    corner = 2.0 ** d if d <= 3 else 1.0
    return float(((1.25 if d <= 3 else 1.6) * corner * k / max(N, 1) * float(np.prod(ext)) / zeta) ** (1.0 / d))


def _table_knn(src, k, dst):
    """mpb200_table_knn: dst = the k best entries of every column of src; returns the number of short columns"""
    nnz, short = _lib.c_i64(0), _lib.c_i64(0)
    _lib.check(_lib.lib().mpb200_table_knn(src.h, int(k), ctypes.byref(dst.h), ctypes.byref(nnz), ctypes.byref(short)))
    dst.nnz, dst.ncols = nnz.value, src.ncols
    return short.value


def _short_columns(table, k):
    """columns of a device table with fewer than k entries (mpb200_table_short_columns)"""
    short = _lib.c_i64(0)
    _lib.check(_lib.lib().mpb200_table_short_columns(table.h, int(k), ctypes.byref(short)))
    return short.value


def _table_union_transpose(a, b, dst):
    nnz = _lib.c_i64(0)
    _lib.check(_lib.lib().mpb200_table_union_transpose(a.h, b.h, ctypes.byref(dst.h), ctypes.byref(nnz)))
    dst.nnz, dst.ncols = nnz.value, a.ncols


class MetricNN(SampleSet):
    """nearneighbors.jl:62-74 for symmetric distances (Euclidean).

    `precompute(r)` plays the role of helper_data_structures + every inball: afterwards
    `self.cache` is an ImmutableNNC and inball/inballF/inballB are column views."""

    def __init__(self, V, dist=None, init=None):
        V = np.ascontiguousarray(V, dtype=np.float64)
        super().__init__(V, dist if dist is not None else Euclidean(), init if init is not None else V[0])
        self.cache = None
        self.table = DeviceTable()

    def build_table(self, r):
        """Device-only: grid build + count + fill; the table stays in HBM. Returns nnz."""
        nnz = _lib.c_i64(0)
        if _is_car(self.dist):
            # ChoppedMetric{ReedsSheppExact}: helper_data_structures = KD-tree over (x, y) (simplecars.jl:42-44),
            # inball = lower-bound candidates + exact metric (nearneighbors.jl:185-198); forward costs only
            # (inballF! and inballB! of a MetricNN are both inball!, nearneighbors.jl:200-203)
            m = self.dist.m
            chop = self.dist.chopval if self.dist.chopval < float("inf") else float(r)
            _lib.check(_lib.lib().mpb200_car_inball_build(self.handle(), m.kind, m.r, float(r), chop,
                                                          ctypes.byref(self.table.h), None, ctypes.byref(nnz), None))
        else:
            _lib.check(_lib.lib().mpb200_inball_build(self.handle(), float(r), ctypes.byref(self.table.h),
                                                      ctypes.byref(nnz)))
        self.table.nnz = nnz.value
        self.table.ncols = self.q1 - self.q0
        self.r = float(r)
        return nnz.value

    def build_table_checked(self, r, CC, SS):
        """Device-only, fused: neighbour table + validity of every stored edge in one pass
        (mpb200_inball_build_checked).  Returns (nnz, checks); bits via fetch_edge_bits()."""
        nnz, checks = _lib.c_i64(0), _lib.c_i64(0)
        d = SS.desc()
        _lib.check(_lib.lib().mpb200_inball_build_checked(self.handle(), float(r), CC.handle(), ctypes.byref(d),
                                                          ctypes.byref(self.table.h), ctypes.byref(nnz),
                                                          ctypes.byref(checks)))
        self.table.nnz = nnz.value
        self.table.ncols = self.q1 - self.q0
        self.r = float(r)
        CC.count += checks.value
        return nnz.value, checks.value

    def fetch_edge_bits(self, table=None):
        table = table or self.table
        bits = self.pool.array(("edge_bits", table.name), (table.nnz + 63) // 64, np.uint64)
        _lib.check(_lib.lib().mpb200_table_fetch_edge_bits(table.h, _lib.ptr(bits)))
        return bits

    def precompute(self, r):
        self.build_table(r)
        D = self.fetch_table(self.table)
        self.cache = ImmutableNNC(D, float(r))
        return self.cache

    def precompute_knn(self, k, r0=None, grow=1.3, max_rounds=40):
        """k-nearest connections (nearneighbors.jl:9-11 exports the names, fmt.jl:17-19 uses them, nothing defines
        them: specification in csrc/knn.cu).  Builds r-ball tables with a growing radius until every column holds at
        least k entries, keeps the k nearest of each (mpb200_table_knn) and forms the mutual neighbourhoods
        (mpb200_table_union_transpose).  Afterwards knn / knnF / knnB / mutualknn* are column views.
        Returns (knn cache, mutual cache); self.r is the radius of the last build (every stored neighbour is within it)."""
        r = self.build_knn(k, r0, grow, max_rounds)
        self.cache_knn = ImmutableNNC(self.fetch_table(self.table_knn, "knn"), float(r))
        self.cache_mknn = ImmutableNNC(self.fetch_table(self.table_mknn, "mknn"), float(r))
        return self.cache_knn, self.cache_mknn

    def build_knn(self, k, r0=None, grow=1.3, max_rounds=40):
        """Device-only part of precompute_knn: the k-nearest table `table_knn` and the mutual table `table_mknn` stay in
        HBM.  Returns the radius of the last r-ball build."""
        N = len(self)
        k = min(int(k), N - 1)
        if k < 1:
            raise ValueError("k-nearest connections need at least two samples")
        if (self.q0, self.q1) != (0, N):
            raise ValueError("k-nearest tables need the full column range (mutual neighbourhoods are a transpose)")
        r = float(r0) if r0 else _knn_radius_guess(self.V, k)
        if not hasattr(self, "table_knn"):
            self.table_knn, self.table_mknn = DeviceTable("knn"), DeviceTable("mknn")
        for _ in range(max_rounds):
            if _is_car(self.dist):
                self.dist.chopval = r                      # setup_steering: the chop value follows the radius
            self.build_table(r)
            if _short_columns(self.table, k) == 0:         # the selection itself runs once, on the final table
                break
            r *= grow
        else:
            raise RuntimeError("k-nearest search did not reach k = %d neighbours per sample" % k)
        _table_knn(self.table, k, self.table_knn)
        _table_union_transpose(self.table_knn, self.table_knn, self.table_mknn)
        self.k = k
        return r

    def car_edges_free(self, CC, SS, fetch=True, table=None):
        return _car_edges_free(self, table if table is not None else self.table, CC, SS, fetch)

    def precompute_checked(self, r, CC, SS):
        """precompute + edge validity through the fused pass -> (ImmutableNNC, edge chunks, checks)"""
        _, checks = self.build_table_checked(r, CC, SS)
        D = self.fetch_table(self.table)
        self.cache = ImmutableNNC(D, float(r))
        return self.cache, self.fetch_edge_bits(), checks

    def close(self):
        self.table.close()
        for name in ("table_knn", "table_mknn"):
            if hasattr(self, name):
                getattr(self, name).close()
        super().close()


class QuasiMetricNN(SampleSet):
    """nearneighbors.jl:76-92 for asymmetric distances (LinearQuadratic): separate forward and
    backward tables.  `precompute(r)` replaces helper_data_structures(V, ::LinearQuadratic)
    (linearquadratic.jl:68-77) and every inballF!/inballB!."""

    def __init__(self, V, dist, init=None):
        V = np.ascontiguousarray(V, dtype=np.float64)
        super().__init__(V, dist, init if init is not None else V[0])
        self.cacheF = self.cacheB = None
        self.tableF, self.tableB = DeviceTable("F"), DeviceTable("B")

    def build_tables(self, r):
        nF, nB = _lib.c_i64(0), _lib.c_i64(0)
        if _is_car(self.dist):                             # ChoppedQuasiMetric{DubinsExact} (simplecars.jl:45-49)
            m = self.dist.m
            chop = self.dist.chopval if self.dist.chopval < float("inf") else float(r)
            _lib.check(_lib.lib().mpb200_car_inball_build(self.handle(), m.kind, m.r, float(r), chop,
                                                          ctypes.byref(self.tableF.h), ctypes.byref(self.tableB.h),
                                                          ctypes.byref(nF), ctypes.byref(nB)))
            for t, n in ((self.tableF, nF), (self.tableB, nB)):
                t.nnz, t.ncols = n.value, self.q1 - self.q0
            self.r = float(r)
            return nF.value, nB.value
        _lib.check(_lib.lib().mpb200_lq_inball_build(self.handle(), self.dist.handle(), float(r),
                                                     ctypes.byref(self.tableF.h), ctypes.byref(self.tableB.h),
                                                     ctypes.byref(nF), ctypes.byref(nB)))
        for t, n in ((self.tableF, nF), (self.tableB, nB)):
            t.nnz, t.ncols = n.value, self.q1 - self.q0
        self.r = float(r)
        return nF.value, nB.value

    def precompute(self, r):
        self.build_tables(r)
        self.cacheF = ImmutableNNC(self.fetch_table(self.tableF, "nnF"), float(r))
        self.cacheB = ImmutableNNC(self.fetch_table(self.tableB, "nnB"), float(r))
        return self.cacheF, self.cacheB

    def precompute_knn(self, k, r0, grow=1.3, max_rounds=30):
        """k-nearest connections under the steering cost: forward / backward cost-ball tables with a growing cost
        radius (from r0) until every column holds k entries, then the k cheapest of each and the mutual forward
        neighbourhoods  knnF(v) U { w : v in knnB(w) }.  Returns (knnF, knnB, mutualF) caches."""
        r = self.build_knn(k, r0, grow, max_rounds)
        self.cache_knnF = ImmutableNNC(self.fetch_table(self.table_knnF, "knnF"), float(r))
        self.cache_knnB = ImmutableNNC(self.fetch_table(self.table_knnB, "knnB"), float(r))
        self.cache_mknnF = ImmutableNNC(self.fetch_table(self.table_mknnF, "mknnF"), float(r))
        return self.cache_knnF, self.cache_knnB, self.cache_mknnF

    def build_knn(self, k, r0, grow=1.3, max_rounds=30):
        """Device-only part of precompute_knn: `table_knnF`, `table_knnB` and `table_mknnF` stay in HBM.  Returns the
        cost radius of the last build."""
        N = len(self)
        k = min(int(k), N - 1)
        r = float(r0)
        if not hasattr(self, "table_knnF"):
            self.table_knnF, self.table_knnB, self.table_mknnF = DeviceTable("knnF"), DeviceTable("knnB"), DeviceTable("mknnF")
        for _ in range(max_rounds):
            if _is_car(self.dist):
                self.dist.chopval = r
            self.build_tables(r)
            if _short_columns(self.tableF, k) == 0 and _short_columns(self.tableB, k) == 0:
                break
            r *= grow
        else:
            raise RuntimeError("k-nearest search did not reach k = %d neighbours per sample" % k)
        _table_knn(self.tableF, k, self.table_knnF)
        _table_knn(self.tableB, k, self.table_knnB)
        _table_union_transpose(self.table_knnF, self.table_knnB, self.table_mknnF)
        self.k = k
        return r

    def car_edges_free(self, CC, SS, fetch=True, table=None):
        return _car_edges_free(self, table if table is not None else self.tableB, CC, SS, fetch)

    def lq_edges_free(self, CC, SS, fetch=True, table=None):
        """validity per stored entry (row y -> column x) of the BACKWARD table (or `table`, e.g. the backward k-nearest
        table): the motion V[y] -> V[x] that fmt.jl:75 asks about; returns (chunks, checks)"""
        d = SS.desc()
        t = table if table is not None else self.tableB
        bits = self.pool.array(("lq_edge_bits", t.name), (t.nnz + 63) // 64, np.uint64) if fetch else None
        checks = _lib.c_i64(0)
        _lib.check(_lib.lib().mpb200_lq_edges_free(self.handle(), t.h, self.dist.handle(), self.r, CC.handle(),
                                                   ctypes.byref(d), _lib.ptr(bits), ctypes.byref(checks)))
        CC.count += checks.value
        return bits, checks.value

    def close(self):
        self.tableF.close()
        self.tableB.close()
        for name in ("table_knnF", "table_knnB", "table_mknnF"):
            if hasattr(self, name):
                getattr(self, name).close()
        super().close()


def addpoints(NN, W):
    """nearneighbors.jl:108-109 -- rebuilds the sample set from scratch, as the reference does."""
    return type(NN)(np.vstack([NN.V, np.atleast_2d(W)]), NN.dist, NN.init)


def inball(NN, v, r, f=None):
    """inball!(NN, v, r[, f]) for a precomputed table (nearneighbors.jl:120,128): v is 1-based
    and global; with sharded tables v must lie in the owned column range."""
    if NN.cache is None:
        NN.precompute(r)
    col = viewcol(NN.cache.D, v - NN.q0)
    return filter_neighborhood(col, f) if f is not None else col


def inballF(NN, v, r, f=None):
    """inballF!(NN, v, r[, f]): nearneighbors.jl:121,128,200-203"""
    if isinstance(NN, MetricNN):
        return inball(NN, v, r, f)
    if NN.cacheF is None:
        NN.precompute(r)
    col = viewcol(NN.cacheF.D, v - NN.q0)
    return filter_neighborhood(col, f) if f is not None else col


def inballB(NN, v, r, f=None):
    """inballB!(NN, v, r[, f]): nearneighbors.jl:122,128,200-203"""
    if isinstance(NN, MetricNN):
        return inball(NN, v, r, f)
    if NN.cacheB is None:
        NN.precompute(r)
    col = viewcol(NN.cacheB.D, v - NN.q0)
    return filter_neighborhood(col, f) if f is not None else col


# ---- k-nearest neighbourhoods (names exported at nearneighbors.jl:9-11; used at fmt.jl:17-19) -----------------
def _need(NN, attr):
    c = getattr(NN, attr, None)
    if c is None:
        raise RuntimeError("call precompute_knn(k) first (k-nearest tables are built for one k)")
    return c


def _served(NN, cache, v, k, f):
    if k != NN.k:
        raise ValueError("the k-nearest tables were built for k = %d" % NN.k)
    col = viewcol(cache.D, v)
    return filter_neighborhood(col, f) if f is not None else col


def knn(NN, v, k, f=None):
    """knn!(NN, v, k[, f]) for a symmetric metric"""
    return _served(NN, _need(NN, "cache_knn"), v, k, f)


def mutualknn(NN, v, k, f=None):
    return _served(NN, _need(NN, "cache_mknn"), v, k, f)


def knnF(NN, v, k, f=None):
    return knn(NN, v, k, f) if isinstance(NN, MetricNN) else _served(NN, _need(NN, "cache_knnF"), v, k, f)


def knnB(NN, v, k, f=None):
    return knn(NN, v, k, f) if isinstance(NN, MetricNN) else _served(NN, _need(NN, "cache_knnB"), v, k, f)


def mutualknnF(NN, v, k, f=None):
    return mutualknn(NN, v, k, f) if isinstance(NN, MetricNN) else _served(NN, _need(NN, "cache_mknnF"), v, k, f)
