"""Known answers of the shortcut restatement (tests/oracle_shortcut.py): the chord without obstacles, a straight input,
a bend around one box corner worked out by hand over its subdivision nodes, L = 1 and L = 2, and a blocked input."""
import math

import numpy as np

import fixtures as fx
from oracle_shortcut import nodes_of, path_cost, shortcut_oracle

BOX = [(np.array([0.25, 0.25]), np.array([0.6875, 0.6875]))]


def _unit(orc):
    return orc.StateSpace([0, 0], [1, 1])


def test_no_obstacles_gives_the_chord(orc):
    Y = np.array([[0.1, 0.1], [0.5, 0.3], [0.2, 0.7], [0.9, 0.9]])
    r = shortcut_oracle(orc, orc.Obstacles2D(fx.EMPTY_2D), _unit(orc), Y, 2)
    assert np.array_equal(r["states"], Y[[0, -1]])
    e = Y[0] - Y[-1]
    assert r["cost"] == math.sqrt(0.0 + e[0] * e[0] + e[1] * e[1])
    assert r["pairs"] == r["segment_checks"] == 7 * 6 // 2


def test_straight_input_gives_its_end_states(orc):
    Y = np.array([[0.125, 0.125], [0.25, 0.125], [0.5, 0.125], [0.875, 0.125]])  # every cost exact: all routes tie
    for k in (1, 2, 4):
        r = shortcut_oracle(orc, orc.Obstacles2D(fx.ISRR_2H), _unit(orc), Y, k)
        assert np.array_equal(r["states"], Y[[0, -1]]) and r["cost"] == 0.75
        assert r["cost"] <= path_cost(Y)


def test_bend_around_one_box_corner(orc):
    # nodes (k = 2): 0 (.5, .125), 1 (.6875, .125), 2 (.875, .125), 3 (.875, .3125), 4 (.875, .5); the box's corner
    # is (.6875, .25).  Only 0 -> 4 crosses the box.  best[4]: via 1 = .1875 + sqrt(.1875^2 + .375^2), via 3 =
    # sqrt(.375^2 + .1875^2) + .1875 (the same sum), via 2 = .75: the tie goes to the smaller a, 1.
    Y = np.array([[0.5, 0.125], [0.875, 0.125], [0.875, 0.5]])
    assert np.array_equal(nodes_of(Y, 2), [[0.5, 0.125], [0.6875, 0.125], [0.875, 0.125], [0.875, 0.3125],
                                           [0.875, 0.5]])
    r = shortcut_oracle(orc, orc.Boxes(BOX), _unit(orc), Y, 2)
    assert np.array_equal(r["states"], [[0.5, 0.125], [0.6875, 0.125], [0.875, 0.5]])
    assert r["cost"] == 0.1875 + math.sqrt(0.17578125) < path_cost(Y) == 0.75
    assert r["pairs"] == r["segment_checks"] == 10
    r1 = shortcut_oracle(orc, orc.Boxes(BOX), _unit(orc), Y, 1)   # no subdivision: nothing to cut
    assert np.array_equal(r1["states"], Y) and r1["cost"] == 0.75 and r1["pairs"] == 3


def test_one_and_two_states(orc):
    O, S = orc.Boxes(BOX), _unit(orc)
    Y1 = np.array([[0.125, 0.875]])
    r = shortcut_oracle(orc, O, S, Y1, 4)
    assert np.array_equal(r["states"], Y1) and r["cost"] == 0.0 and r["pairs"] == r["segment_checks"] == 0
    Y2 = np.array([[0.125, 0.125], [0.125, 0.875]])
    r = shortcut_oracle(orc, O, S, Y2, 2)
    assert np.array_equal(r["states"], Y2) and r["cost"] == 0.75 and r["pairs"] == 3


def test_blocked_input_comes_back_unchanged(orc):
    Y = np.array([[0.125, 0.125], [0.125, 0.5], [0.875, 0.5], [0.875, 0.875]])  # the middle edge crosses the box
    r = shortcut_oracle(orc, orc.Boxes(BOX), _unit(orc), Y, 2)
    assert np.array_equal(r["states"], Y) and r["cost"] == math.inf
    assert r["pairs"] == 7 * 6 // 2
