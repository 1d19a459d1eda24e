"""FMT* over GPU-precomputed neighbour and validity tables.

Host restatement of src/planners/fmt.jl:4-119 (`fmtstar!`): the heap-ordered wavefront and the
tree bookkeeping stay on the host exactly as north_star prescribes; what changes is where its
three hot calls are served from:
  nearF / nearB (fmt.jl:70,72)    -> column views of the ImmutableNNC tables built by K1/K2 or K5
  F[i] = is_free_state (:31-36)   -> one batched K6 call
  is_free_motion(V[y], V[x]) (:75)-> a bit lookup in the edge-validity table built by K7/K8/K9,
                                     aligned with the backward table (row y, column x)
The neighbour iteration order (ascending index), findmin's first-minimum tie-break and the
"collision_checks" metadata (lookups actually consumed, one per segment test the lazy reference
would have run) are preserved.
"""
import math
import time

import numpy as np

from .linearquadratic import LinearQuadratic, setup_steering
from .simplecars import is_car_metric
from .nearneighbors import MetricNN
from .problems import MPSolution, goal_mask, sample_free
from .statespaces import Euclidean, states_free, volume


class PriorityQueue:
    """Collections.PriorityQueue of Julia 0.5 (base/collections.jl; the reference uses it at fmt.jl:51,78,86): a binary
    min-heap of key => priority pairs in an array with an index dictionary.  Restated -- not heapq with (cost, x)
    tuples -- because the order in which EQUAL priorities leave the queue is a property of this particular heap
    (percolate_up stops at a parent that is not strictly larger; percolate_down prefers the left child unless the right
    one is strictly smaller), and FMT*'s expansion order, hence its tree, depends on it when costs tie (lattices)."""

    def __init__(self):
        self.xs = []          # (key, priority)
        self.index = {}       # key -> 1-based position

    def __len__(self):
        return len(self.xs)

    def _up(self, i):
        xs = self.xs
        x = xs[i - 1]
        while i > 1:
            j = i >> 1
            if x[1] < xs[j - 1][1]:
                self.index[xs[j - 1][0]] = i
                xs[i - 1] = xs[j - 1]
                i = j
            else:
                break
        self.index[x[0]] = i
        xs[i - 1] = x

    def _down(self, i):
        xs = self.xs
        n = len(xs)
        x = xs[i - 1]
        while 2 * i <= n:
            l, r = 2 * i, 2 * i + 1
            j = l if (r > n or xs[l - 1][1] < xs[r - 1][1]) else r
            if xs[j - 1][1] < x[1]:
                self.index[xs[j - 1][0]] = i
                xs[i - 1] = xs[j - 1]
                i = j
            else:
                break
        self.index[x[0]] = i
        xs[i - 1] = x

    def __setitem__(self, key, value):
        """pq[key] = value: enqueue!, or re-prioritise an existing key"""
        if key in self.index:
            i = self.index[key]
            old = self.xs[i - 1][1]
            self.xs[i - 1] = (key, value)
            if old < value:
                self._down(i)
            else:
                self._up(i)
        else:
            self.xs.append((key, value))
            self.index[key] = len(self.xs)
            self._up(len(self.xs))

    def dequeue(self):
        x = self.xs[0]
        y = self.xs.pop()
        if self.xs:
            self.xs[0] = y
            self.index[y[0]] = 1
            self._down(1)
        del self.index[x[0]]
        return x[0]


def fmt_radius(N, d, rm, free_volume_ub):
    """fmt.jl:37-41"""
    return rm * 2 * (1 / d * free_volume_ub / (math.pi ** (d / 2) / math.gamma(d / 2 + 1)) * math.log(N) / N) ** (1 / d)


def _bits_to_bool(chunks, n):
    return np.unpackbits(np.ascontiguousarray(chunks).view(np.uint8), bitorder="little")[:n].astype(bool)


def fmtstar(P, N=None, rm=1.0, connections="R", r=0.0, ensure_goal_ct=1, init_idx=1, checkpts=True, seed=0,
            edge_checks="table", k=None):
    """fmtstar!(P, N; rm, connections, r, ensure_goal_ct, init_idx, checkpts) -> (status, cost, elapsed)

    edge_checks = "table": the validity of EVERY stored edge is precomputed in one pass (K7/K8/K9) and fmt.jl:75
    becomes a bit lookup -- the right trade when the table is large and the GPU pass costs microseconds per
    million edges.  edge_checks = "lazy": wavefront-batched lazy checking (SURVEY 8f.2) -- no edge table; the
    candidate connections (y_min, x) of ONE expansion of z are independent of each other (H and C only change
    after the loop, fmt.jl:69-84), so they are checked in one batched device call per expansion and the device
    work equals what FMT* consumes ("collision_checks").  Both modes return the identical tree, path and cost."""
    t_start = time.perf_counter()
    N = len(P.V) if N is None else N
    P.CC.count = 0
    if connections not in ("R", "K"):
        raise ValueError("Connection type must be radial (:R) or k-nearest (:K)")
    # connections = :K: nearF = mutualknnF!, nearB = knnB! (fmt.jl:17-19).  The reference exports those names
    # (nearneighbors.jl:9-11) but never defines them, so :K throws there; here they follow the specification of
    # csrc/knn.cu (k nearest by stored value, ties to the smaller index; mutual = knnF U transpose(knnB)).
    knn_mode = connections == "K"
    SS, CC = P.SS, P.CC
    if r > 0:
        setup_steering(SS, r)
    if not states_free(P.init, CC, SS)[0]:
        P.status = "failed"                               # fmt.jl:24-29
        P.solution = MPSolution(P.status, math.inf, time.perf_counter() - t_start, {})
        return math.inf
    free_volume_ub = sample_free(P, N - len(P.V), ensure_goal_ct=ensure_goal_ct, seed=seed) if N > len(P.V) else volume(SS)
    NN = P.V
    V = NN.V
    if r == 0:
        r = fmt_radius(N, SS.dim, rm, free_volume_ub)
        setup_steering(SS, r)
    if k is None:                                          # fmt.jl:6
        k = min(int(math.ceil((2 * rm) ** SS.dim * (math.e / SS.dim) * math.log(N))), N - 1)

    # ---- the batched precompute that replaces the lazy per-call hot path -----------------------
    if edge_checks not in ("table", "lazy"):
        raise ValueError("edge_checks must be 'table' or 'lazy'")
    lazy = edge_checks == "lazy"
    lq = isinstance(SS.dist, LinearQuadratic)
    car = is_car_metric(SS.dist)
    ebits = None
    if knn_mode and (lq or (car and not SS.dist.symmetric)):
        cF, cB, cM = NN.precompute_knn(k, r)               # cost radius grows from r until every column holds k
        r = cB.r
        setup_steering(SS, r)                              # the steering horizon of the waypoint checks = the last radius
        NN.r = r
        DF, DB = cM.D, cB.D
        if not lazy:
            ebits, _ = (NN.car_edges_free if car else NN.lq_edges_free)(CC, SS, table=NN.table_knnB)
    elif knn_mode and car:                                 # Reeds-Shepp MetricNN: knnF = knnB = knn (forward lengths)
        cK, cM = NN.precompute_knn(k, r)
        r = cK.r
        setup_steering(SS, r)
        NN.r = r
        DF, DB = cM.D, cK.D
        if not lazy:
            ebits, _ = NN.car_edges_free(CC, SS, table=NN.table_knn)
    elif knn_mode:
        cK, cM = NN.precompute_knn(k)
        DF, DB = cM.D, cK.D
        if not lazy:
            ebits, _ = NN.edges_free(NN.table_knn, CC, SS)
    elif car:
        if SS.dist.symmetric:                              # MetricNN: inballF! = inballB! = inball! (forward costs)
            DF = DB = NN.precompute(r).D
        else:
            cF, cB = NN.precompute(r)
            DF, DB = cF.D, cB.D
        if not lazy:
            ebits, _ = NN.car_edges_free(CC, SS)
    elif lq:
        cF, cB = NN.precompute(r)
        DF, DB = cF.D, cB.D
        if not lazy:
            ebits, _ = NN.lq_edges_free(CC, SS)
    elif lazy:
        DF = DB = NN.precompute(r).D
    else:
        cache, ebits, _ = NN.precompute_checked(r, CC, SS)   # K1 + K2 with K7/K8 fused
        DF = DB = cache.D
    lookups_before = CC.count
    CC.count = 0                                          # the table build is not what FMT* "asked"
    evalid = _bits_to_bool(ebits, DB.nnz) if not lazy else None
    if lazy:
        from .linearquadratic import lq_motions_free
        from .simplecars import car_motions_free
        from .statespaces import segments_free
    F = _bits_to_bool(NN.points_free(CC, SS), N) if checkpts else np.ones(N, dtype=bool)
    is_goal = goal_mask(V, P.goal, SS)

    # per-edge number of segment tests the lazy checker would have run (CC.count parity):
    # Euclidean edges: 1 if the first endpoint is inside the state bounds, else 0
    inb = np.all((SS.lo <= V) & (V <= SS.hi), axis=1)

    A = np.zeros(N, dtype=np.int64)
    Wm = np.ones(N, dtype=bool)
    H = np.zeros(N, dtype=bool)
    C = np.zeros(N)
    if not np.all(V[init_idx - 1] == P.init):
        raise RuntimeError("P.V[init_idx] must be the init state (fmt.jl:48-66)")
    Wm[init_idx - 1] = False
    H[init_idx - 1] = True
    heap = PriorityQueue()                               # HHeap (fmt.jl:51); init_idx is dequeued at once (:67)
    z = init_idx
    fcp, frv, fnz = DF.colptr, DF.rowval, DF.nzval
    bcp, brv, bnz = DB.colptr, DB.rowval, DB.nzval
    checks = 0
    device_batches = 0
    while not is_goal[z - 1]:
        H_new = []
        fs = frv[fcp[z - 1] - 1:fcp[z] - 1]
        todo = []                                          # (x, y_min, c_min, stored entry) of this expansion, in x order
        for x in fs[Wm[fs - 1]]:                           # nearF(V, z, r, W): unvisited, ascending
            x = int(x)
            if checkpts and not F[x - 1]:
                continue
            lo, hi = bcp[x - 1] - 1, bcp[x] - 1
            ys = brv[lo:hi]
            keep = H[ys - 1]                               # nearB(V, x, r, H): open neighbours
            cand = ys[keep]
            if cand.size == 0:                             # cannot happen for consistent F/B tables
                continue
            costs = C[cand - 1] + bnz[lo:hi][keep]
            j = int(np.argmin(costs))                      # findmin: first minimum
            c_min, y_min = float(costs[j]), int(cand[j])
            e = lo + int(np.flatnonzero(keep)[j])          # stored entry (row y_min, column x)
            if lq or car:
                checks += 1                                # counted per motion; segments in metadata below
            else:
                checks += int(inb[y_min - 1])
            todo.append((x, y_min, c_min, e))
        if lazy and todo:                                  # ONE batched device call for the whole expansion
            ys_ = np.fromiter((t[1] for t in todo), dtype=np.int64) - 1
            xs_ = np.fromiter((t[0] for t in todo), dtype=np.int64) - 1
            ok = (car_motions_free if car else lq_motions_free if lq else segments_free)(V[ys_], V[xs_], CC, SS)
            device_batches += 1
        for t_i, (x, y_min, c_min, e) in enumerate(todo):
            if (ok[t_i] if lazy else evalid[e]):             # is_free_motion(V[y_min], V[x], CC, SS)
                A[x - 1] = y_min
                C[x - 1] = c_min
                heap[x] = c_min                            # HHeap[x] = c_min (fmt.jl:78)
                H_new.append(x)
                Wm[x - 1] = False
        if H_new:
            H[np.asarray(H_new) - 1] = True
        H[z - 1] = False
        if len(heap):
            z = heap.dequeue()
        else:
            break

    sol = [z]
    costs = [C[z - 1]]
    while sol[0] != 1:                                     # fmt.jl:92-101 (assumes init_idx == 1)
        sol.insert(0, int(A[sol[0] - 1]))
        if sol[0] == 0:
            costs.insert(0, 0.0)
            break
        costs.insert(0, C[sol[0] - 1])
    solved = bool(is_goal[z - 1])
    P.status = "solved" if solved else "failed"
    CC.count = checks
    meta = {
        "radius_multiplier": rm, "collision_checks": checks, "num_samples": N, "cost": float(C[z - 1]),
        "cumcost": costs, "planner": "FMTstar", "solved": solved, "tree": A, "path": sol, "r": r,
        "precomputed_edge_checks": int(lookups_before), "edge_checks": edge_checks,
        "connections": connections, "k": (k if knn_mode else None),
        "device_edge_batches": device_batches,
    }
    P.solution = MPSolution(P.status, float(C[z - 1]), time.perf_counter() - t_start, meta)
    return P.status, P.solution.cost, P.solution.elapsed


def _gmt_roadmap(P, N, rm, connections, r, ensure_goal_ct, checkpts, seed, k, lazy):
    """The roadmap GMT* plans over, left on the device: sample_free up to N samples, the radius (fmt.jl:37-41) and
    steering, the forward and backward tables of the connection type, the edge bits of the backward table (none when
    lazy) and the point bits (checkpts).  -> dict(NN, DF, DB, r, k, lookups_before, lq, car, knn_mode)"""
    SS, CC = P.SS, P.CC
    knn_mode = connections == "K"
    free_volume_ub = sample_free(P, N - len(P.V), ensure_goal_ct=ensure_goal_ct, seed=seed) if N > len(P.V) else volume(SS)
    NN = P.V
    if r == 0:
        r = fmt_radius(N, SS.dim, rm, free_volume_ub)
        setup_steering(SS, r)
    if k is None:
        k = min(int(math.ceil((2 * rm) ** SS.dim * (math.e / SS.dim) * math.log(N))), N - 1)

    # ---- the same tables and bits as fmtstar(edge_checks="table"), left on the device (lazy: no bits) ---------
    lq = isinstance(SS.dist, LinearQuadratic)
    car = is_car_metric(SS.dist)
    if knn_mode and (lq or (car and not SS.dist.symmetric)):
        r = NN.build_knn(k, r)
        setup_steering(SS, r)
        NN.r = r
        DF, DB = NN.table_mknnF, NN.table_knnB
        if not lazy:
            (NN.car_edges_free if car else NN.lq_edges_free)(CC, SS, fetch=False, table=DB)
    elif knn_mode and car:
        r = NN.build_knn(k, r)
        setup_steering(SS, r)
        NN.r = r
        DF, DB = NN.table_mknn, NN.table_knn
        if not lazy:
            NN.car_edges_free(CC, SS, fetch=False, table=DB)
    elif knn_mode:
        NN.build_knn(k)
        DF, DB = NN.table_mknn, NN.table_knn
        if not lazy:
            NN.edges_free(DB, CC, SS, fetch=False)
    elif car and SS.dist.symmetric:
        NN.build_table(r)
        DF = DB = NN.table
        if not lazy:
            NN.car_edges_free(CC, SS, fetch=False)
    elif car or lq:
        NN.build_tables(r)
        DF, DB = NN.tableF, NN.tableB
        if not lazy:
            (NN.car_edges_free if car else NN.lq_edges_free)(CC, SS, fetch=False)
    elif lazy:
        NN.build_table(r)
        DF = DB = NN.table
    else:
        NN.build_table_checked(r, CC, SS)
        DF = DB = NN.table
    lookups_before = CC.count
    CC.count = 0
    if checkpts:
        NN.points_free(CC, SS, fetch=False)
    return dict(NN=NN, DF=DF, DB=DB, r=r, k=k, lookups_before=lookups_before, lq=lq, car=car, knn_mode=knn_mode)


def _gmt_edges(rm, CC):
    """the lazy motion check of the roadmap's metric (mpb200_gmt_edges)"""
    from . import _lib
    NN = rm["NN"]
    if rm["car"]:
        m_ = NN.dist.m
        return _lib.GmtEdges(_lib.GMT_EDGES_CAR, CC.handle(), None, 0.0, m_.kind, m_.r, m_.s)
    if rm["lq"]:
        return _lib.GmtEdges(_lib.GMT_EDGES_LQ, CC.handle(), NN.dist.handle(), NN.r, 0, 0.0, 0.0)
    return _lib.GmtEdges(_lib.GMT_EDGES_STRAIGHT, CC.handle(), None, 0.0, 0, 0.0, 0.0)


def _goal_chunks(V, goal, SS):
    """the goal mask of V as host BitVector chunks (ceil(N/64) uint64 words)"""
    chunks = np.zeros((len(V) + 63) // 64 * 8, dtype=np.uint8)
    packed = np.packbits(goal_mask(V, goal, SS), bitorder="little")
    chunks[:len(packed)] = packed
    return chunks.view(np.uint64)


def _gmt_check_args(connections, lams, edge_checks):
    if connections not in ("R", "K"):
        raise ValueError("Connection type must be radial (:R) or k-nearest (:K)")
    if not all(lam >= 0 for lam in lams):
        raise ValueError("lam must be a non-negative number")
    if edge_checks not in ("table", "lazy"):
        raise ValueError("edge_checks must be 'table' or 'lazy'")


def _gmt_meta(rm, res, sol, C, tree, checks, lam, connections, edge_checks, device_ms, N, rmult):
    return {
        "radius_multiplier": rmult, "collision_checks": checks, "num_samples": N, "cost": float(res.cost),
        "cumcost": None if C is None else [float(C[v - 1]) for v in sol], "planner": "GMTstar",
        "solved": bool(res.solved), "tree": tree, "path": sol, "r": rm["r"],
        "precomputed_edge_checks": int(rm["lookups_before"]), "edge_checks": edge_checks,
        "connections": connections, "k": (rm["k"] if rm["knn_mode"] else None), "device_edge_batches": 0,
        "lambda": lam, "iterations": int(res.iterations), "expansions": int(res.expansions), "device_ms": device_ms,
        "costs": C, "checks": int(res.checks), "checks_in_bounds": int(res.checks_in_bounds),
        "grid_blocks": int(res.grid_blocks),
    }


def gmtstar(P, N=None, rm=1.0, connections="R", r=0.0, lam=1.0, ensure_goal_ct=1, init_idx=1, checkpts=True, seed=0,
            k=None, edge_checks="table"):
    """Group-marching FMT* (GMT*; Ichter, Schmerling & Pavone 2017) planned on the device -> (status, cost, elapsed)

    Sets the problem up exactly as fmtstar does (radius, steering, sample_free, goal mask), builds the tables and
    validity bits with the device-only calls and plans over them in one cooperative kernel (mpb200_gmt_plan): each
    iteration expands, all at once, every open vertex whose cost is within lam * r of the cheapest one.  No table
    crosses PCIe; the path, tree and costs come back.  At lam = 0 (and no two open vertices of equal cost) the tree,
    path, cost and "collision_checks" equal fmtstar's.  Specification: include/mpb200.h, DESIGN.md section 10b.

    edge_checks = "table": every stored edge of the backward table is checked in one pass before planning and the
    planner reads its bit.  edge_checks = "lazy": no edge pass; the planning kernel runs the motion check of the one
    entry each candidate connects through (mpb200_gmt_plan_lazy), so only the motions the plan uses are checked.  Both
    modes return the identical tree, path, cost and counters; lazy adds "segment_checks", the segment tests it ran."""
    from . import _lib
    import ctypes

    t_start = time.perf_counter()
    N = len(P.V) if N is None else N
    P.CC.count = 0
    _gmt_check_args(connections, [lam], edge_checks)
    lazy = edge_checks == "lazy"
    SS, CC = P.SS, P.CC
    if r > 0:
        setup_steering(SS, r)
    if not states_free(P.init, CC, SS)[0]:
        P.status = "failed"
        P.solution = MPSolution(P.status, math.inf, time.perf_counter() - t_start, {})
        return math.inf
    rmap = _gmt_roadmap(P, N, rm, connections, r, ensure_goal_ct, checkpts, seed, k, lazy)
    NN, DF, DB = rmap["NN"], rmap["DF"], rmap["DB"]
    V = NN.V
    if not np.all(V[init_idx - 1] == P.init):
        raise RuntimeError("P.V[init_idx] must be the init state (fmt.jl:48-66)")
    goal_chunks = _goal_chunks(V, P.goal, SS)

    space = SS.desc()
    desc = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(goal_chunks), init_idx, float(lam) * float(rmap["r"]),
                        int(bool(checkpts)), ctypes.pointer(space))
    res = _lib.GmtResult()
    tree = np.empty(N, dtype=np.int64)
    C = np.empty(N, dtype=np.float64)
    path = np.empty(N, dtype=np.int64)
    lib = _lib.lib()
    if lazy:
        edges = _gmt_edges(rmap, CC)
        segment_checks = _lib.c_i64(0)
        _lib.check(lib.mpb200_gmt_plan_lazy(NN.handle(), ctypes.byref(desc), ctypes.byref(edges), ctypes.byref(res),
                                            ctypes.byref(segment_checks), _lib.ptr(path), N, _lib.ptr(tree),
                                            _lib.ptr(C)))
    else:
        _lib.check(lib.mpb200_gmt_plan(NN.handle(), ctypes.byref(desc), ctypes.byref(res), _lib.ptr(path), N,
                                       _lib.ptr(tree), _lib.ptr(C)))
    device_ms = lib.mpb200_last_ms_of(_lib.OP_PLAN, 0)
    sol = [int(v) for v in path[:res.path_len]]
    # fmtstar counts a Euclidean check only when y lies in the state bounds (the lazy checker's segment count)
    checks = int(res.checks) if (rmap["lq"] or rmap["car"]) else int(res.checks_in_bounds)
    P.status = "solved" if res.solved else "failed"
    CC.count = checks
    meta = _gmt_meta(rmap, res, sol, C, tree, checks, lam, connections, edge_checks, device_ms, N, rm)
    if lazy:
        meta["segment_checks"] = int(segment_checks.value)
    P.solution = MPSolution(P.status, float(res.cost), time.perf_counter() - t_start, meta)
    return P.status, P.solution.cost, P.solution.elapsed


def gmtstar_batch(P, inits, goals, lam=1.0, N=None, rm=1.0, connections="R", r=0.0, ensure_goal_ct=1, checkpts=True,
                  seed=0, k=None, edge_checks="table", trees=True):
    """A batch of GMT* queries over one roadmap -> [MPSolution], one per query

    The roadmap is set up exactly as gmtstar sets it up (sample 1 = P.init, P.goal's goal samples, radius, steering,
    tables, bits); then every query q, from sample inits[q] (1-based) to goals[q] (a goal object: its mask is goal_mask)
    at width lam[q] * r (lam: a scalar or one value per query), is planned in one cooperative launch
    (mpb200_gmt_plan_batch).  Each query's solution equals what gmtstar would return for it over the same roadmap;
    a query whose init sample is not free is "failed" without a plan.  Metadata: gmtstar's keys plus "query" (its
    position in the batch) and "batch_size"; "device_ms" is the time of the batch's kernel.  trees=False skips the
    nq x N tree and cost copies ("tree", "costs" and "cumcost" are None)."""
    from . import _lib
    import ctypes

    t_start = time.perf_counter()
    inits = [int(i) for i in inits]
    goals = list(goals)
    nq = len(inits)
    if nq == 0 or len(goals) != nq:
        raise ValueError("inits and goals must be non-empty and of the same length")
    lams = [float(x) for x in np.broadcast_to(np.asarray(lam, dtype=np.float64), (nq,))]
    N = len(P.V) if N is None else N
    P.CC.count = 0
    _gmt_check_args(connections, lams, edge_checks)
    if not all(1 <= i <= N for i in inits):
        raise ValueError("inits must be sample indices 1..N")
    lazy = edge_checks == "lazy"
    SS, CC = P.SS, P.CC
    if r > 0:
        setup_steering(SS, r)
    rmap = _gmt_roadmap(P, N, rm, connections, r, ensure_goal_ct, checkpts, seed, k, lazy)
    NN, DF, DB = rmap["NN"], rmap["DF"], rmap["DB"]
    V = NN.V
    free = states_free(V[np.asarray(inits) - 1], CC, SS)      # fmt.jl:24-29, per query
    planned = [q for q in range(nq) if free[q]]
    n = len(planned)
    space = SS.desc()
    chunks = [_goal_chunks(V, goals[q], SS) for q in planned]
    descs = (_lib.GmtDesc * max(n, 1))()
    for j, q in enumerate(planned):
        descs[j] = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(chunks[j]), inits[q], lams[q] * float(rmap["r"]),
                                int(bool(checkpts)), ctypes.pointer(space))
    res = (_lib.GmtResult * max(n, 1))()
    # a path can be N long, so each row holds N; np.empty only reserves address space and the library writes path_len
    # entries of a row, so what becomes resident is the pages those paths touch (one 2 MB page a row with huge pages)
    paths = np.empty((n, N), dtype=np.int64)
    tree = np.empty((n, N), dtype=np.int64) if trees else None
    C = np.empty((n, N), dtype=np.float64) if trees else None
    segs = np.zeros(max(n, 1), dtype=np.int64)
    lib = _lib.lib()
    device_ms = 0.0
    if n:
        edges = ctypes.byref(_gmt_edges(rmap, CC)) if lazy else None
        _lib.check(lib.mpb200_gmt_plan_batch(NN.handle(), descs, n, edges, res, _lib.ptr(segs) if lazy else None,
                                             _lib.ptr(paths), N, _lib.ptr(tree), _lib.ptr(C)))
        device_ms = lib.mpb200_last_ms_of(_lib.OP_PLAN, 0)
    elapsed = time.perf_counter() - t_start
    out = [MPSolution("failed", math.inf, elapsed, {"query": q, "batch_size": nq}) for q in range(nq)]
    total_checks = 0
    for j, q in enumerate(planned):
        rq = res[j]
        sol = [int(v) for v in paths[j, :rq.path_len]]
        checks = int(rq.checks) if (rmap["lq"] or rmap["car"]) else int(rq.checks_in_bounds)
        total_checks += checks
        meta = _gmt_meta(rmap, rq, sol, None if C is None else C[j], None if tree is None else tree[j], checks,
                         lams[q], connections, edge_checks, device_ms, N, rm)
        if lazy:
            meta["segment_checks"] = int(segs[j])
        meta["query"], meta["batch_size"] = q, nq
        out[q] = MPSolution("solved" if rq.solved else "failed", float(rq.cost), elapsed, meta)
    CC.count = total_checks
    return out


def prmstar(P, N=None, rm=1.0, connections="R", r=0.0, ensure_goal_ct=1, init_idx=1, checkpts=True, seed=0, k=None):
    """PRM*: the shortest path over the roadmap, planned on the device -> (status, cost, elapsed)

    Sets the problem and the roadmap up exactly as gmtstar(edge_checks="table") does (sample_free, radius, steering,
    tables, edge bits, point bits), then finds, in one cooperative kernel (mpb200_sssp_plan), the cheapest path from
    sample init_idx to the goal region over every collision-free edge of the backward table: a cost no FMT*-family
    planner over the same roadmap can beat.  The tree and costs come back for every vertex no costlier than the goal
    (every reachable vertex when the plan fails); the others have parent 0 and cost inf.  Specification:
    include/mpb200.h, DESIGN.md section 10d.  Metadata: "planner" = "PRMstar", "path", "tree", "costs", "r", "k",
    "rounds", "levels", "reached", "device_ms" and the roadmap keys gmtstar reports."""
    from . import _lib
    import ctypes

    t_start = time.perf_counter()
    N = len(P.V) if N is None else N
    P.CC.count = 0
    _gmt_check_args(connections, [0.0], "table")
    SS, CC = P.SS, P.CC
    if r > 0:
        setup_steering(SS, r)
    if not states_free(P.init, CC, SS)[0]:
        P.status = "failed"
        P.solution = MPSolution(P.status, math.inf, time.perf_counter() - t_start, {})
        return math.inf
    rmap = _gmt_roadmap(P, N, rm, connections, r, ensure_goal_ct, checkpts, seed, k, False)
    NN, DF, DB = rmap["NN"], rmap["DF"], rmap["DB"]
    V = NN.V
    if not np.all(V[init_idx - 1] == P.init):
        raise RuntimeError("P.V[init_idx] must be the init state (fmt.jl:48-66)")
    goal_chunks = _goal_chunks(V, P.goal, SS)
    space = SS.desc()
    desc = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(goal_chunks), init_idx, 0.0, int(bool(checkpts)), ctypes.pointer(space))
    res = _lib.SsspResult()
    tree = np.empty(N, dtype=np.int64)
    C = np.empty(N, dtype=np.float64)
    path = np.empty(N, dtype=np.int64)
    lib = _lib.lib()
    _lib.check(lib.mpb200_sssp_plan(NN.handle(), ctypes.byref(desc), ctypes.byref(res), _lib.ptr(path), N,
                                    _lib.ptr(tree), _lib.ptr(C)))
    device_ms = lib.mpb200_last_ms_of(_lib.OP_PLAN, 0)
    sol = [int(v) for v in path[:res.path_len]]
    P.status = "solved" if res.solved else "failed"
    meta = {
        "radius_multiplier": rm, "num_samples": N, "cost": float(res.cost), "cumcost": [float(C[v - 1]) for v in sol],
        "planner": "PRMstar", "solved": bool(res.solved), "tree": tree, "path": sol, "costs": C, "r": rmap["r"],
        "k": (rmap["k"] if rmap["knn_mode"] else None), "connections": connections,
        "precomputed_edge_checks": int(rmap["lookups_before"]), "rounds": int(res.rounds), "levels": int(res.levels),
        "reached": int(res.reached), "device_ms": device_ms, "grid_blocks": int(res.grid_blocks),
    }
    P.solution = MPSolution(P.status, float(res.cost), time.perf_counter() - t_start, meta)
    return P.status, P.solution.cost, P.solution.elapsed


def prmstar_batch(P, inits, goals, N=None, rm=1.0, connections="R", r=0.0, ensure_goal_ct=1, checkpts=True, seed=0,
                  k=None, trees=True):
    """A batch of PRM* queries over one roadmap -> [MPSolution], one per query

    The roadmap is set up exactly as prmstar sets it up (sample 1 = P.init, P.goal's goal samples, radius, steering,
    tables, edge bits, point bits); then every query q, from sample inits[q] (1-based) to goals[q] (a goal object: its
    mask is goal_mask), is planned in one cooperative launch (mpb200_sssp_plan_batch).  Each query's solution equals
    what prmstar would return for it over the same roadmap; a query whose init sample is not free is "failed" without a
    plan.  Metadata: prmstar's keys plus "query" (its position in the batch) and "batch_size"; "device_ms" is the time
    of the batch's kernel.  trees=False skips the nq x N tree and cost copies ("tree", "costs" and "cumcost" are
    None)."""
    from . import _lib
    import ctypes

    t_start = time.perf_counter()
    inits = [int(i) for i in inits]
    goals = list(goals)
    nq = len(inits)
    if nq == 0 or len(goals) != nq:
        raise ValueError("inits and goals must be non-empty and of the same length")
    N = len(P.V) if N is None else N
    P.CC.count = 0
    _gmt_check_args(connections, [0.0], "table")
    if not all(1 <= i <= N for i in inits):
        raise ValueError("inits must be sample indices 1..N")
    SS, CC = P.SS, P.CC
    if r > 0:
        setup_steering(SS, r)
    rmap = _gmt_roadmap(P, N, rm, connections, r, ensure_goal_ct, checkpts, seed, k, False)
    NN, DF, DB = rmap["NN"], rmap["DF"], rmap["DB"]
    V = NN.V
    free = states_free(V[np.asarray(inits) - 1], CC, SS)      # fmt.jl:24-29, per query
    planned = [q for q in range(nq) if free[q]]
    n = len(planned)
    space = SS.desc()
    chunks = [_goal_chunks(V, goals[q], SS) for q in planned]
    descs = (_lib.GmtDesc * max(n, 1))()
    for j, q in enumerate(planned):
        descs[j] = _lib.GmtDesc(DF.h, DB.h, _lib.ptr(chunks[j]), inits[q], 0.0, int(bool(checkpts)),
                                ctypes.pointer(space))
    res = (_lib.SsspResult * max(n, 1))()
    paths = np.empty((n, N), dtype=np.int64)                  # rows as gmtstar_batch: only path_len entries are written
    tree = np.empty((n, N), dtype=np.int64) if trees else None
    C = np.empty((n, N), dtype=np.float64) if trees else None
    lib = _lib.lib()
    device_ms = 0.0
    if n:
        _lib.check(lib.mpb200_sssp_plan_batch(NN.handle(), descs, n, res, _lib.ptr(paths), N, _lib.ptr(tree),
                                              _lib.ptr(C)))
        device_ms = lib.mpb200_last_ms_of(_lib.OP_PLAN, 0)
    elapsed = time.perf_counter() - t_start
    out = [MPSolution("failed", math.inf, elapsed, {"query": q, "batch_size": nq}) for q in range(nq)]
    for j, q in enumerate(planned):
        rq = res[j]
        sol = [int(v) for v in paths[j, :rq.path_len]]
        meta = {
            "radius_multiplier": rm, "num_samples": N, "cost": float(rq.cost),
            "cumcost": None if C is None else [float(C[j, v - 1]) for v in sol], "planner": "PRMstar",
            "solved": bool(rq.solved), "tree": None if tree is None else tree[j], "path": sol,
            "costs": None if C is None else C[j], "r": rmap["r"], "k": (rmap["k"] if rmap["knn_mode"] else None),
            "connections": connections, "precomputed_edge_checks": int(rmap["lookups_before"]),
            "rounds": int(rq.rounds), "levels": int(rq.levels), "reached": int(rq.reached), "device_ms": device_ms,
            "grid_blocks": int(rq.grid_blocks), "query": q, "batch_size": nq,
        }
        out[q] = MPSolution("solved" if rq.solved else "failed", float(rq.cost), elapsed, meta)
    return out


def shortcut_paths(P, paths=None, subdivisions=4):
    """The cheapest collision-free route through each path's subdivided waypoints (mpb200_shortcut_paths) -> [dict]

    paths: a list whose items are either a 1-D sequence of 1-based sample indices into P.V (the "path" of any solution,
    including each gmtstar_batch result) or an (L, d) array of states; default [P.solution.metadata["path"]].  Each
    edge is cut into `subdivisions` pieces; over the resulting waypoints, every pair a < b whose straight motion is free
    under P.CC and P.SS is an edge of a DAG with the Euclidean cost, and the cheapest route from the first to the last
    waypoint comes back (ties to the longest jump).  Not the reference's shortcut / adaptive_shortcut!: specified in
    include/mpb200.h and DESIGN.md section 10c.  For a planner's solution under the same P.CC and P.SS the returned cost
    is never above the planned one, and shortcutting a result again never raises its cost.  A path that is not free
    comes back unchanged with cost inf.
    Per path: {"states": (L', d) array, "cost": float, "pairs": waypoint pairs, "segment_checks": segment tests run};
    the segment tests are added to P.CC.count, as segments_free does.  All paths go to the device in one call."""
    from . import _lib
    import ctypes

    SS, CC = P.SS, P.CC
    if not isinstance(SS.dist, Euclidean):
        raise ValueError("shortcut_paths needs straight-line motions: Reeds-Shepp, Dubins and linear-quadratic spaces "
                         "connect states by curves whose cost is defined only up to the steering radius")
    if int(subdivisions) != subdivisions or subdivisions < 1:
        raise ValueError("subdivisions must be an integer >= 1")
    if paths is None:
        sol = getattr(P, "solution", None)
        if sol is None or sol.status != "solved":
            raise ValueError("P has no solved path to shortcut")
        paths = [sol.metadata["path"]]
    d = SS.dim
    V = P.V.V if hasattr(P.V, "V") else None
    states = []
    for p in paths:
        a = np.asarray(p)
        if a.ndim == 1 and a.size and np.issubdtype(a.dtype, np.integer):
            if V is None or np.any(a < 1) or np.any(a > len(V)):
                raise ValueError("path indices must be sample indices 1..N of P.V")
            a = V[a - 1]
        elif a.ndim == 2 and a.shape[0] >= 1 and a.shape[1] == d and np.issubdtype(a.dtype, np.number):
            a = a.astype(np.float64)
        else:
            raise ValueError("each path must be non-empty: 1-based sample indices or an (L, %d) array of states" % d)
        states.append(np.ascontiguousarray(a, dtype=np.float64))
    n = len(states)
    if n == 0:
        raise ValueError("no paths given")
    offsets = np.zeros(n + 1, dtype=np.int64)
    offsets[1:] = np.cumsum([len(s) for s in states])
    Y = np.ascontiguousarray(np.vstack(states))
    k = int(subdivisions)
    cap = max((len(s) - 1) * k + 1 for s in states)
    out = np.empty((n, cap, d), dtype=np.float64)
    out_len = np.empty(n, dtype=np.int64)
    costs = np.empty(n, dtype=np.float64)
    pairs = np.empty(n, dtype=np.int64)
    segs = np.empty(n, dtype=np.int64)
    space = SS.desc()
    _lib.check(_lib.lib().mpb200_shortcut_paths(_lib.ptr(Y), _lib.ptr(offsets), n, d, CC.handle(), ctypes.byref(space),
                                                k, _lib.ptr(out), cap, _lib.ptr(out_len), _lib.ptr(costs),
                                                _lib.ptr(pairs), _lib.ptr(segs)))
    CC.count += int(segs.sum())
    return [{"states": out[q, :out_len[q]].copy(), "cost": float(costs[q]), "pairs": int(pairs[q]),
             "segment_checks": int(segs[q])} for q in range(n)]
