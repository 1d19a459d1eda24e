"""CPU restatement of mpb200_shortcut_paths, written from its specification (include/mpb200.h, DESIGN.md section 10c) and
independent of the product code: nodes and costs in numpy (squares summed coordinate by coordinate), visibility from one
call of the oracle's edges_free_csc, the minimum as a loop over b with np.argmin.  Test infrastructure."""
import numpy as np


def nodes_of(Y, k):
    """the (L - 1) k + 1 nodes: Y[i] at i k, Y[i] + t (Y[i+1] - Y[i]) with t = m / k in between (one rounding each)"""
    Y = np.asarray(Y, dtype=np.float64)
    L, d = Y.shape
    X = np.empty(((L - 1) * k + 1, d))
    X[::k] = Y
    for m in range(1, k):
        t = np.float64(m) / np.float64(k)
        X[m::k] = Y[:-1] + t * (Y[1:] - Y[:-1])
    return X


def cost_matrix(X):
    """cost[a, b] = sqrt(sum_c (X[a, c] - X[b, c])^2), the sum in index order"""
    s = np.zeros((len(X), len(X)))
    for c in range(X.shape[1]):
        e = X[:, None, c] - X[None, :, c]
        s = s + e * e
    return np.sqrt(s)


def visibility(orc, obs, space, X):
    """free[a, b] for a < b (node a bounds-checked, node b not) and the segment tests run, in one edges_free_csc call
    over the CSC whose column b holds the rows 0..b-1"""
    M = len(X)
    counts = np.arange(M, dtype=np.int64)
    colptr = np.concatenate([[1], 1 + np.cumsum(counts)]).astype(np.int64)
    rowval = np.concatenate([np.arange(1, b + 1, dtype=np.int64) for b in range(M)]) if M > 1 else np.zeros(0, np.int64)
    ok, checks = orc.edges_free_csc(obs, space, X, colptr, rowval)
    free = np.zeros((M, M), dtype=bool)
    for b in range(1, M):
        free[:b, b] = ok[colptr[b] - 1:colptr[b + 1] - 1].astype(bool)
    return free, checks


def shortcut_oracle(orc, obs, space, Y, k):
    """-> dict(states, cost, pairs, segment_checks) of one path Y (L x d) with k subdivisions"""
    Y = np.asarray(Y, dtype=np.float64)
    X = nodes_of(Y, k)
    M = len(X)
    free, checks = visibility(orc, obs, space, X)
    C = cost_matrix(X)
    best = np.full(M, np.inf)
    pred = np.full(M, -1)
    best[0] = 0.0
    for b in range(1, M):
        a = np.flatnonzero(free[:b, b])
        if a.size == 0:
            continue
        v = best[a] + C[a, b]
        j = int(np.argmin(v))                               # first minimum: the smallest a
        if np.isfinite(v[j]):
            best[b], pred[b] = v[j], a[j]
    if np.isfinite(best[M - 1]):
        chain = [M - 1]
        while chain[-1] != 0:
            chain.append(int(pred[chain[-1]]))
        states, cost = X[chain[::-1]], float(best[M - 1])
    else:
        states, cost = Y.copy(), float("inf")
    return dict(states=states, cost=cost, pairs=M * (M - 1) // 2, segment_checks=int(checks))


def path_cost(Y):
    """the edge costs of Y summed in path order (the planner's C[goal] for a planned path)"""
    c = 0.0
    for i in range(len(Y) - 1):
        s = 0.0
        for j in range(Y.shape[1]):
            e = Y[i, j] - Y[i + 1, j]
            s = s + e * e
        c = c + float(np.sqrt(s))
    return c
