"""Test infrastructure: group-marching FMT* (GMT*; Ichter, Schmerling & Pavone 2017) restated on the CPU from its
specification (include/mpb200.h, DESIGN.md section 10b) over the oracle's neighbourhoods and lazy edge checks, written
independently of the product's planner and kernel.  Each iteration works on whole vertex sets: the group, the
candidates and the new open vertices are computed from the state at the start of the iteration and applied at its end."""
import numpy as np

W, H, CLOSED = 0, 1, 2


def gmt_oracle(N, is_goal, neighborsF, neighborsB, point_free, edge_free, w, init=1, checkpts=True, in_bounds=None):
    """N samples (1-based); neighborsF/B(v) -> (inds 1-based ascending, costs); point_free(i0) -> bool;
    edge_free(y0, x0) -> (bool, segment checks the lazy checker runs); w = lambda * r; in_bounds(y0) -> bool.
    Returns dict(solved, goal, cost, path, tree, costs, iterations, expansions, checks, checks_in_bounds, seg_checks)."""
    is_goal = np.asarray(is_goal, dtype=bool)
    F = np.array([point_free(i) for i in range(N)], dtype=bool) if checkpts else np.ones(N, dtype=bool)
    C = np.zeros(N)
    A = np.zeros(N, dtype=np.int64)
    state = np.full(N, W, dtype=np.int8)
    state[init - 1] = H
    out = dict(iterations=0, expansions=0, checks=0, checks_in_bounds=0, seg_checks=0)
    while True:
        openv = np.flatnonzero(state == H)
        if openv.size == 0:
            return dict(out, solved=False, goal=0, cost=float("inf"), path=[], tree=A, costs=C)
        thr = np.float64(C[openv].min()) + np.float64(w)
        group = openv[C[openv] <= thr]
        goals = [int(g) for g in group if is_goal[g]]
        if goals:
            g = min(goals, key=lambda v: (C[v], v))
            path = [g + 1]
            while path[0] != init:
                path.insert(0, int(A[path[0] - 1]))
            return dict(out, solved=True, goal=g + 1, cost=float(C[g]), path=path, tree=A, costs=C)
        cand = set()
        for g in group:
            for x in neighborsF(int(g) + 1)[0]:
                x0 = int(x) - 1
                if state[x0] == W and F[x0]:
                    cand.add(x0)
        joined = []
        for x0 in sorted(cand):
            inds, costs = neighborsB(x0 + 1)
            best = None
            for y, cy in zip(inds, costs):
                y0 = int(y) - 1
                if state[y0] != H:
                    continue
                c = np.float64(C[y0]) + np.float64(cy)
                if best is None or c < best[0]:      # strict: the first entry in storage order wins a tie
                    best = (c, y0)
            if best is None:                          # no open neighbour in the backward table: skip x
                continue
            c, y0 = best
            out["checks"] += 1
            if in_bounds is not None and in_bounds(y0):
                out["checks_in_bounds"] += 1
            ok, n = edge_free(y0, x0)
            out["seg_checks"] += n
            if ok:
                joined.append((x0, y0, c))
        for x0, y0, c in joined:
            C[x0], A[x0], state[x0] = c, y0 + 1, H
        state[group] = CLOSED
        out["iterations"] += 1
        out["expansions"] += int(group.size)
