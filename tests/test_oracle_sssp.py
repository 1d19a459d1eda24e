"""The CPU restatement of the roadmap-optimal plan (tests/oracle_sssp.py) on hand-built CSC graphs whose answers are
worked out by hand, and on random graphs against a plain Bellman-Ford restatement.  No GPU needed."""
import numpy as np
import pytest

from oracle_sssp import sssp_numpy, sssp_oracle

INF = float("inf")


def csc(N, edges):
    """edges: (y, x, w) 1-based, an entry of row y in column x; columns stored with rows ascending (stable)"""
    edges = sorted(edges, key=lambda t: (t[1], t[0]))
    colptr = np.concatenate([[1], 1 + np.cumsum(np.bincount([x - 1 for _, x, _ in edges], minlength=N))])
    rowval = np.array([y for y, _, _ in edges], dtype=np.int64)
    nzval = np.array([w for _, _, w in edges], dtype=np.float64)
    return colptr, rowval, nzval


def plan(N, edges, goals, init=1, free=None, cleared=()):
    cp, rv, nz = csc(N, edges)
    bits = np.ones(len(rv), dtype=bool)
    for y, x in cleared:
        e = cp[x - 1] - 1 + int(np.flatnonzero(rv[cp[x - 1] - 1:cp[x] - 1] == y)[0])
        bits[e] = False
    free = np.ones(N, dtype=bool) if free is None else np.asarray(free, dtype=bool)
    g = np.zeros(N, dtype=bool)
    g[np.asarray(goals, dtype=np.int64) - 1] = True
    a = sssp_oracle(N, cp, rv, nz, bits, free, g, init)
    b = sssp_numpy(N, cp, rv, nz, bits, free, g, init)
    for k in a:
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    return a


def both(y, x, w):
    return [(y, x, w), (x, y, w)]


def test_diamond_ties_go_to_storage_order():
    r = plan(4, [(1, 2, 1.0), (1, 3, 1.0), (2, 4, 1.0), (3, 4, 1.0)], [4])
    assert r["solved"] and r["cost"] == 2.0 and r["path"] == [1, 2, 4] and r["goal"] == 4
    assert list(r["tree"]) == [0, 1, 1, 2] and r["levels"] == 3 and r["reached"] == 4


def test_duplicate_vertices_joined_by_zero_cost_edges_give_an_acyclic_tree():
    # 2 and 3 are the same state: zero-cost entries both ways; only 3 is entered from the init
    r = plan(4, both(2, 3, 0.0) + [(1, 3, 1.0), (2, 4, 1.0), (3, 4, 1.0)], [4])
    assert r["cost"] == 2.0 and list(r["costs"]) == [0.0, 1.0, 1.0, 2.0]
    # the tight edges 2 -> 3 and 3 -> 2 form a cycle; depth decides: h(3) = 1 through row 1, h(2) = 2 through row 3
    assert list(r["tree"]) == [0, 3, 1, 3] and r["path"] == [1, 3, 4] and r["levels"] == 3


def test_absorbed_addition_does_not_close_a_parent_cycle():
    # init 4; 4 -> 2 costs 1; 1 <-> 2 cost 1e-17, absorbed: d(1) = d(2) = 1.0.  Column 2's first tight entry is row 1,
    # whose parent would be 2: the depth rule takes row 4 instead.
    r = plan(4, [(4, 2, 1.0), (2, 1, 1e-17), (1, 2, 1e-17)], [1], init=4)
    assert 1.0 + 1e-17 == 1.0
    assert r["solved"] and r["cost"] == 1.0 and r["goal"] == 1
    assert list(r["tree"]) == [2, 4, 0, 0] and r["path"] == [4, 2, 1]


def test_diagonal_entry_is_not_an_edge():
    r = plan(3, [(1, 2, 1.0), (2, 2, 0.0), (2, 3, 1.0)], [3])
    assert r["path"] == [1, 2, 3] and list(r["tree"]) == [0, 1, 2]
    r = plan(2, [(2, 2, 0.0), (1, 1, 0.0)], [2])
    assert not r["solved"] and r["reached"] == 1


def test_unreachable_goal_fails_with_the_full_tree():
    edges = both(1, 2, 1.0) + both(2, 3, 0.5) + both(1, 3, 2.0)
    r = plan(5, edges + both(4, 5, 1.0), [5])
    assert not r["solved"] and r["cost"] == INF and r["goal"] == 0 and r["path"] == []
    assert list(r["costs"]) == [0.0, 1.0, 1.5, INF, INF] and list(r["tree"]) == [0, 1, 2, 0, 0]
    assert r["reached"] == 3 and r["levels"] == 3
    r0 = plan(5, edges + both(4, 5, 1.0), [])
    assert list(r0["costs"]) == list(r["costs"]) and list(r0["tree"]) == list(r["tree"])


def test_init_as_goal():
    # 2 duplicates the init 3 (zero cost both ways) and is a goal with a smaller index: the init is the goal
    r = plan(4, both(2, 3, 0.0) + both(3, 4, 1.0), [2, 3], init=3)
    assert r["solved"] and r["cost"] == 0.0 and r["path"] == [3] and r["goal"] == 3
    assert r["reached"] == 2 and list(r["tree"]) == [0, 3, 0, 0] and list(r["costs"]) == [INF, 0.0, 0.0, INF]


def test_checkpts_excludes_a_vertex():
    edges = [(1, 2, 1.0), (2, 4, 1.0), (1, 3, 1.5), (3, 4, 1.5)]
    assert plan(4, edges, [4])["path"] == [1, 2, 4]
    r = plan(4, edges, [4], free=[True, False, True, True])
    assert r["path"] == [1, 3, 4] and r["cost"] == 3.0 and r["costs"][1] == INF


def test_cleared_edge_bit():
    edges = [(1, 2, 1.0), (2, 4, 1.0), (1, 3, 1.5), (3, 4, 1.5)]
    r = plan(4, edges, [4], cleared=[(2, 4)])
    assert r["path"] == [1, 3, 4] and r["cost"] == 3.0 and r["costs"][1] == 1.0 and r["tree"][1] == 1


def test_cut_off_masks_vertices_costlier_than_the_goal():
    edges = [(1, 2, 1.0), (2, 3, 1.0), (3, 4, 1.0), (1, 5, 2.0), (5, 6, 0.5)]
    r = plan(6, edges, [3])
    assert r["cost"] == 2.0 and r["reached"] == 4                        # 1, 2, 3 and 5 (d = 2 = d*, a tie)
    assert list(r["costs"]) == [0.0, 1.0, 2.0, INF, 2.0, INF] and list(r["tree"]) == [0, 1, 2, 0, 1, 0]


def _bellman_ford(N, cp, rv, nz, bits, free, init):
    d = [INF] * N
    d[init - 1] = 0.0
    for _ in range(N):
        changed = False
        for x in range(N):
            if not free[x]:
                continue
            for e in range(cp[x] - 1, cp[x + 1] - 1):
                y = rv[e] - 1
                if bits[e] and y != x and d[y] + nz[e] < d[x]:
                    d[x] = d[y] + nz[e]
                    changed = True
        if not changed:
            break
    return np.array(d)


@pytest.mark.parametrize("seed", range(12))
def test_random_graphs_match_bellman_ford_and_the_folds(seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    N = int(rng.integers(2, 40))
    M = int(rng.integers(0, 5 * N))
    pairs = {(int(rng.integers(1, N + 1)), int(rng.integers(1, N + 1))) for _ in range(M)}
    # costs with ties, zeros and absorbed additions
    pool = np.array([0.0, 1e-17, 0.1, 0.2, 0.3, 1.0, 1.0 / 3.0, 0.7])
    edges = [(y, x, float(pool[rng.integers(len(pool))])) for y, x in sorted(pairs)]
    cp, rv, nz = csc(N, edges)
    bits = rng.random(len(rv)) < 0.85
    free = rng.random(N) < 0.9
    g = rng.random(N) < (0.1 if seed % 3 else 0.0)
    init = int(rng.integers(1, N + 1))
    r = sssp_oracle(N, cp, rv, nz, bits, free, g, init)
    b = sssp_numpy(N, cp, rv, nz, bits, free, g, init)
    for k in r:
        assert np.array_equal(np.asarray(r[k]), np.asarray(b[k])), k
    d = _bellman_ford(N, cp, rv, nz, bits, free, init)
    in_r = np.isfinite(r["costs"])
    assert np.array_equal(r["costs"][in_r], d[in_r])
    if r["solved"]:
        assert np.all(d[~in_r] > r["cost"]) and r["cost"] == min(d[g])
    else:
        assert np.all(~np.isfinite(d[~in_r])) and not np.isfinite(d[g]).any()
    for x in np.flatnonzero(in_r):                                      # each parent chain folds to its cost
        chain = [x + 1]
        while chain[0] != init:
            chain.insert(0, int(r["tree"][chain[0] - 1]))
            assert len(chain) <= N
        c = 0.0
        for y, x1 in zip(chain[:-1], chain[1:]):
            lo, hi = cp[x1 - 1] - 1, cp[x1] - 1
            e = lo + int(np.flatnonzero(rv[lo:hi] == y)[0])
            c = c + float(nz[e])
        assert c == r["costs"][x]
