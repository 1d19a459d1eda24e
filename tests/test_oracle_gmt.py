"""The CPU restatement of GMT* (tests/oracle_gmt.py): equal to FMT* (tests/oracle_fmt.py) at w = 0 on config C1, and
the known trees, iteration counts and corner cases of hand-built graphs."""
import numpy as np
import pytest

import fixtures as fx
from oracle_fmt import fmt_oracle
from oracle_gmt import gmt_oracle


def _c1(orc, N, obst):
    """config C1: sample 1 = init (.1, .1), last = goal (.9, .9), the rest uniform and free"""
    if obst == "BOXES2D":
        O = orc.Boxes(fx.BOXES2D)
    else:
        O = orc.Obstacles2D(fx.ALL_2D[obst])
    So = orc.StateSpace([0, 0], [1, 1])
    cand = fx.uniform_samples(3 * N, 2, 20240601)
    cand = cand[orc.states_free(O, So, cand)][:N - 2]
    return np.vstack([[0.1, 0.1], cand, [0.9, 0.9]]), O, So


@pytest.mark.parametrize("obst", ["ISRR_2H", "BOXES2D"])
def test_gmt_at_zero_width_is_fmt_on_c1(orc, obst):
    N = 1000
    V, O, So = _c1(orc, N, obst)
    r = fx.fmt_radius(N, 2)
    T = orc.KDTree(V).rball(r)
    col = lambda v: (T[1][T[0][v - 1] - 1:T[0][v] - 1], T[2][T[0][v - 1] - 1:T[0][v] - 1])

    def edge(y0, x0):
        ok, n = orc.motions_free_straight(O, So, V[y0:y0 + 1], V[x0:x0 + 1])
        return bool(ok[0]), n

    free = lambda i: bool(orc.states_free(O, So, V[i:i + 1])[0])
    goal = np.all(V == [0.9, 0.9], axis=1)
    ref = fmt_oracle(V, goal, col, col, free, edge)
    got = gmt_oracle(N, goal, col, col, free, edge, 0.0, in_bounds=lambda y0: bool(np.all((0 <= V[y0]) & (V[y0] <= 1))))
    assert ref["solved"] and got["solved"]
    assert got["path"] == ref["path"] and np.array_equal(got["tree"], ref["tree"])
    assert got["cost"] == ref["cost"]
    assert got["seg_checks"] == got["checks_in_bounds"] == ref["checks"]
    assert got["iterations"] == got["expansions"]            # one vertex per group
    # a wider group: fewer iterations, a cost no better than FMT*'s on the same samples
    wide = gmt_oracle(N, goal, col, col, free, edge, 1.0 * r)
    assert wide["solved"] and wide["iterations"] < got["iterations"] and wide["cost"] >= ref["cost"] * (1 - 1e-12)


def _graph(N, edges):
    """hand-built tables from {(y, x): cost} (1-based): DF column z lists x with z -> x, DB column x lists y with y -> x"""
    F = {v: [] for v in range(1, N + 1)}
    B = {v: [] for v in range(1, N + 1)}
    for (y, x), c in edges.items():
        F[y].append((x, c))
        B[x].append((y, c))
    col = lambda T: (lambda v: (np.array([i for i, _ in sorted(T[v])], dtype=np.int64),
                                np.array([c for _, c in sorted(T[v])], dtype=np.float64)))
    return col(F), col(B)


def _run(N, edges, goal, w, blocked=(), free=None):
    nF, nB = _graph(N, edges)
    is_goal = np.zeros(N, dtype=bool)
    is_goal[[g - 1 for g in goal]] = True
    return gmt_oracle(N, is_goal, nF, nB, (lambda i: True) if free is None else free,
                      lambda y0, x0: ((y0 + 1, x0 + 1) not in blocked, 1), w)


# 1 -> 2 -> 5 -> 4 is cheap (2.0) but 5 opens only after 2 is expanded; 3 -> 4 is dear (13.0)
DETOUR = {(1, 2): 1.0, (1, 3): 3.0, (2, 5): 0.5, (5, 4): 0.5, (3, 4): 10.0}


@pytest.mark.parametrize("w,cost,path,iters,exps", [
    (0.0, 2.0, [1, 2, 5, 4], 3, 3),     # FMT*: 1, 2, 5 expanded one at a time; 4 connects through 5
    (1.0, 2.0, [1, 2, 5, 4], 3, 3),     # thr = 1 + 1 keeps 3 (C = 3) out of the second group
    (5.0, 13.0, [1, 3, 4], 3, 4),       # {2, 3} expanded together: 4 connects through 3 before 5 is open
    (1e9, 13.0, [1, 3, 4], 2, 3),       # every open vertex in G: {1}, {2, 3}, then {4, 5} holds the goal
])
def test_gmt_hand_graph_known_trees(w, cost, path, iters, exps):
    got = _run(5, DETOUR, [4], w)
    assert got["solved"] and got["cost"] == cost and got["path"] == path
    assert got["iterations"] == iters and got["expansions"] == exps
    assert got["checks"] == 4
    assert got["tree"][3] == path[-2]


def test_gmt_tied_costs_both_enter_the_group():
    edges = {(1, 2): 1.0, (1, 3): 1.0, (2, 4): 1.0, (3, 5): 1.0}
    got = _run(5, edges, [5], 0.0)
    assert got["solved"] and got["cost"] == 2.0 and got["path"] == [1, 3, 5]
    assert got["iterations"] == 2 and got["expansions"] == 3      # {1}, then {2, 3} together
    assert list(got["tree"]) == [0, 1, 1, 2, 3]


def test_gmt_candidate_without_open_backward_neighbour_is_skipped():
    # 2 is in DF[1] but DB[2] only holds 3 (k-nearest tables need not be transposes): skipped, no check counted,
    # reached later from 3
    nF = lambda v: {1: ([2, 3], [1.0, 1.0]), 2: ([], []), 3: ([2], [1.0])}[v]
    nB = lambda v: {1: ([], []), 2: ([3], [1.0]), 3: ([1], [1.0])}[v]
    got = gmt_oracle(3, [False, True, False], nF, nB, lambda i: True, lambda y0, x0: (True, 1), 0.0)
    assert got["solved"] and got["path"] == [1, 3, 2] and got["cost"] == 2.0
    assert got["checks"] == 2 and got["iterations"] == 2


def test_gmt_blocked_edge_leaves_the_vertex_unvisited():
    edges = {(1, 2): 1.0, (1, 3): 2.0, (2, 4): 1.0, (3, 4): 1.5}
    got = _run(4, edges, [4], 0.0, blocked={(2, 4)})
    assert got["solved"] and got["path"] == [1, 3, 4] and got["cost"] == 3.5
    assert got["checks"] == 4                      # 2, 3, then 4 from 2 (blocked), then 4 again from 3


def test_gmt_point_validity_excludes_candidates():
    got = _run(5, DETOUR, [4], 0.0, free=lambda i: i != 4)      # sample 5 in collision
    assert got["solved"] and got["path"] == [1, 3, 4] and got["cost"] == 13.0


def test_gmt_init_is_goal():
    got = _run(5, DETOUR, [1, 4], 0.0)
    assert got["solved"] and got["cost"] == 0.0 and got["path"] == [1]
    assert got["iterations"] == 0 and got["expansions"] == 0 and got["checks"] == 0


def test_gmt_unreachable_goal_fails():
    got = _run(6, DETOUR, [6], 0.0)
    assert not got["solved"] and got["cost"] == float("inf") and got["path"] == []
    assert got["iterations"] == 5 and got["expansions"] == 5
