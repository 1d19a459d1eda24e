"""Test infrastructure: the roadmap-optimal plan (PRM*; mpb200_sssp_plan) restated on the CPU from its specification
(include/mpb200.h, DESIGN.md section 10d) over a backward table DB (1-based CSC), its edge bits and the point bits,
written independently of the kernel.  sssp_oracle runs Dijkstra with heapq for the costs, then a BFS over the tight
edges and the parent rule; sssp_numpy is the same specification vectorised over frontiers (Bellman-Ford rounds) for
tables too large for a Python heap.  Every addition is one Python float (IEEE binary64, round to nearest) add."""
import heapq

import numpy as np


def _graph_entries(colptr, rowval, ebits, free):
    """-> (row y, column x, entry e) 0-based of every graph edge y -> x, in storage order"""
    cp, rv = np.asarray(colptr, dtype=np.int64) - 1, np.asarray(rowval, dtype=np.int64) - 1
    col = np.repeat(np.arange(len(cp) - 1), np.diff(cp))
    ok = np.asarray(ebits, dtype=bool) & (rv != col) & np.asarray(free, dtype=bool)[col]
    e = np.flatnonzero(ok)
    return rv[e], col[e], e


def _finish(N, d, colptr, rowval, nzval, ebits, free, is_goal, init, h):
    """the outputs from the costs d and the depths h (-1 = not in R): goal, parents, masks"""
    is_goal = np.asarray(is_goal, dtype=bool)
    gs = np.flatnonzero(is_goal)
    dstar = min((d[g] for g in gs), default=np.inf)
    in_r = (d <= dstar) & np.isfinite(d)
    cp, rv, nz = np.asarray(colptr) - 1, np.asarray(rowval) - 1, np.asarray(nzval, dtype=np.float64)
    eb, fr = np.asarray(ebits, dtype=bool), np.asarray(free, dtype=bool)
    tree = np.zeros(N, dtype=np.int64)
    for x in np.flatnonzero(in_r):
        if x == init - 1:
            continue
        for e in range(cp[x], cp[x + 1]):          # storage order: the first tight entry one level up
            y = int(rv[e])
            if eb[e] and y != x and fr[x] and h[y] == h[x] - 1 and float(d[y]) + float(nz[e]) == float(d[x]):
                tree[x] = y + 1
                break
        assert tree[x] != 0, x
    costs = np.where(in_r, d, np.inf)
    out = dict(reached=int(in_r.sum()), levels=int(h[in_r].max()) + 1, tree=tree, costs=costs)
    if not np.isfinite(dstar):
        return dict(out, solved=False, goal=0, cost=float("inf"), path=[])
    goal = init - 1 if is_goal[init - 1] else int(min(gs[d[gs] == dstar]))
    path = [goal + 1]
    while path[0] != init:
        path.insert(0, int(tree[path[0] - 1]))
    assert len(path) == h[goal] + 1
    return dict(out, solved=True, goal=goal + 1, cost=float(dstar), path=path)


def sssp_oracle(N, colptr, rowval, nzval, ebits, free, is_goal, init=1):
    """DB as 1-based CSC (colptr N+1, rowval, nzval); ebits bool[nnz]; free bool[N] (all True without checkpts);
    is_goal bool[N]; init 1-based.  -> dict(solved, goal, cost, path, tree, costs, reached, levels)"""
    ys, xs, es = _graph_entries(colptr, rowval, ebits, free)
    nz = np.asarray(nzval, dtype=np.float64)
    out = [[] for _ in range(N)]
    for y, x, e in zip(ys.tolist(), xs.tolist(), es.tolist()):
        out[y].append((x, float(nz[e])))
    d = [float("inf")] * N
    d[init - 1] = 0.0
    heap = [(0.0, init - 1)]
    done = [False] * N
    while heap:
        c, y = heapq.heappop(heap)
        if done[y]:
            continue
        done[y] = True
        for x, w in out[y]:
            nd = c + w
            if nd < d[x]:
                d[x] = nd
                heapq.heappush(heap, (nd, x))
    d = np.array(d)
    gs = np.flatnonzero(np.asarray(is_goal, dtype=bool))
    dstar = min((d[g] for g in gs), default=np.inf)
    in_r = (d <= dstar) & np.isfinite(d)
    h = np.full(N, -1, dtype=np.int64)
    h[init - 1] = 0
    frontier, level = [init - 1], 0
    while frontier:
        nxt = []
        for y in frontier:
            for x, w in out[y]:
                if in_r[x] and h[x] == -1 and d[y] + w == d[x]:
                    h[x] = level + 1
                    nxt.append(x)
        frontier, level = nxt, level + 1
    assert np.all(h[in_r] >= 0), "a vertex of R is not reached over the tight edges"
    return _finish(N, d, colptr, rowval, nzval, ebits, free, is_goal, init, h)


def sssp_numpy(N, colptr, rowval, nzval, ebits, free, is_goal, init=1):
    """sssp_oracle vectorised: frontier Bellman-Ford for the costs, a frontier BFS for the depths, the parent rule on
    whole arrays.  Same outputs (the fixed point is unique)."""
    ys, xs, es = _graph_entries(colptr, rowval, ebits, free)
    ws = np.asarray(nzval, dtype=np.float64)[es]
    order = np.argsort(ys, kind="stable")
    ys, xs, es, ws = ys[order], xs[order], es[order], ws[order]
    start = np.searchsorted(ys, np.arange(N + 1))

    def out_edges(front):
        cnt = start[front + 1] - start[front]
        idx = np.repeat(start[front] - np.cumsum(np.r_[0, cnt[:-1]]), cnt) + np.arange(cnt.sum())
        return idx

    d = np.full(N, np.inf)
    d[init - 1] = 0.0
    front = np.array([init - 1])
    while front.size:
        idx = out_edges(front)
        cand = d[ys[idx]] + ws[idx]
        old = d.copy()
        np.minimum.at(d, xs[idx], cand)
        front = np.flatnonzero(d < old)
    gs = np.flatnonzero(np.asarray(is_goal, dtype=bool))
    dstar = d[gs].min() if gs.size else np.inf
    in_r = (d <= dstar) & np.isfinite(d)
    h = np.full(N, -1, dtype=np.int64)
    h[init - 1] = 0
    front, level = np.array([init - 1]), 0
    while front.size:
        idx = out_edges(front)
        x = xs[idx]
        tight = in_r[x] & (h[x] == -1) & (d[ys[idx]] + ws[idx] == d[x])
        front = np.unique(x[tight])
        h[front] = level + 1
        level += 1
    assert np.all(h[in_r] >= 0)
    # parents: per column, the first entry in storage order that is tight and one level up
    cp = np.asarray(colptr, dtype=np.int64) - 1
    rv = np.asarray(rowval, dtype=np.int64) - 1
    col = np.repeat(np.arange(N), np.diff(cp))
    nz = np.asarray(nzval, dtype=np.float64)
    ok = (np.asarray(ebits, dtype=bool) & (rv != col) & np.asarray(free, dtype=bool)[col] & in_r[col] &
          (h[rv] == h[col] - 1) & (h[col] > 0) & (d[rv] + nz == d[col]))
    e = np.flatnonzero(ok)
    cols, first = np.unique(col[e], return_index=True)
    tree = np.zeros(N, dtype=np.int64)
    tree[cols] = rv[e[first]] + 1
    costs = np.where(in_r, d, np.inf)
    out = dict(reached=int(in_r.sum()), levels=int(h[in_r].max()) + 1, tree=tree, costs=costs)
    if not np.isfinite(dstar):
        return dict(out, solved=False, goal=0, cost=float("inf"), path=[])
    goal = init - 1 if is_goal[init - 1] else int(gs[d[gs] == dstar].min())
    path = [goal + 1]
    while path[0] != init:
        path.insert(0, int(tree[path[0] - 1]))
    return dict(out, solved=True, goal=goal + 1, cost=float(dstar), path=path)
