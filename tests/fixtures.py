"""Obstacle-set fixtures as raw constructor inputs (test/obstaclesets/2D.jl:3-42, ND.jl:1-14),
written independently of the product package so that oracle and product tables can be
compared, plus the seeded synthetic-input generators of SURVEY 8(d)."""
import math

import numpy as np


def box2d(xr, yr):  # SAT2D.jl:53-56
    return ("polygon", [(xr[0], yr[0]), (xr[1], yr[0]), (xr[1], yr[1]), (xr[0], yr[1])])


ISRR_2H = ("compound", [
    box2d([.0, .16], [.36, .5]), box2d([.4, .5], [.19, .35]), box2d([.22, .46], [.57, .75]),
    box2d([.75, 1.], [.64, .77]), box2d([.22, .8], [.34, .51])])
TRI_BALLS = ("compound", [
    ("polygon", [(.3, .3), (.7, .3), (.5, .65)]),
    ("circle", (.3, .3), .15), ("circle", (.7, .3), .15), ("circle", (.5, .65), .15)])
ISRR_POLY = ("compound", [
    ("polygon", [(.0, .25), (.27, .28), (.17, .4), (.0, .4)]),
    ("polygon", [(.5, .2), (.2, .5), (.25, .7), (.4, .8), (.6, .8), (.7, .5)]),
    ("polygon", [(.55, .2), (.75, .5), (.85, .5), (.85, .2)]),
    ("circle", (.9, .65), .1)])
ISRR_POLY_WITH_SPIKE = ("compound", [
    ("polygon", [(.0, .25), (.27, .28), (.17, .4), (.0, .4)]),
    ("polygon", [(.5, .2), (.2, .5), (.25, .7), (.4, .8), (.6, .8), (.7, .5)]),
    ("polygon", [(.55, .2), (.75, .5), (.85, .5), (.85, .2)]),
    ("polygon", [(.3, .6), (.15, .85), (.4, .6)]),
    ("circle", (.9, .65), .1)])
EMPTY_2D = ("compound", [])
ALL_2D = {"ISRR_2H": ISRR_2H, "TRI_BALLS": TRI_BALLS, "ISRR_POLY": ISRR_POLY,
          "ISRR_POLY_WITH_SPIKE": ISRR_POLY_WITH_SPIKE, "EMPTY_2D": EMPTY_2D}

BOXES2D = [np.array(b) for b in ([[0., 0.16], [0.36, 0.5]], [[0.4, 0.5], [0.19, 0.35]], [[0.22, 0.46], [0.57, 0.75]],
                                 [[0.75, 1.], [0.64, 0.77]], [[0.22, 0.8], [0.34, 0.51]])]
BOXES3D = [np.array(r, dtype=float).T.copy() for r in (
    [[0.25, 0, 0], [.3, .4, 1]], [[0.25, .6, 0], [.3, 1, 1]], [[0.25, .4, 0], [.3, .6, .25]],
    [[0.25, .4, .33], [.3, .6, .7]], [[0.25, .4, .85], [.3, .6, 1]], [[0.7, 0, 0], [.75, 1, .3]],
    [[0.7, 0, .5], [.75, 1, 1]], [[0.7, 0, .3], [.75, .2, .5]], [[0.7, .4, .3], [.75, .5, .5]],
    [[0.7, .7, .3], [.75, 1, .5]])]


def product_shape(mp, spec):
    """Build the product-side shape tree from a raw spec."""
    if spec[0] == "compound":
        return mp.Compound2D([product_shape(mp, s) for s in spec[1]])
    if spec[0] == "circle":
        return mp.Circle(spec[1], spec[2])
    return mp.Polygon(spec[1])


def fmt_radius(N, d, rm=1.0, vol=1.0):
    """fmt.jl:37-41"""
    return rm * 2 * (1 / d * vol / (math.pi ** (d / 2) / math.gamma(d / 2 + 1)) * math.log(N) / N) ** (1 / d)


def uniform_samples(N, d, seed):
    return np.random.Generator(np.random.PCG64(seed)).random((N, d))


def lattice_cloud(rng, n, d, step, lo, hi):
    """points on the lattice step * Z^d inside [lo, hi]^d (exactly representable: differences and squares are exact)"""
    k0, k1 = int(np.ceil(lo / step)), int(np.floor(hi / step))
    return rng.integers(k0, k1 + 1, size=(n, d)).astype(np.float64) * step


def random_hyperboxes(M, d, seed, init=0.1, goal=0.9):
    """SURVEY 8(d) C3: centre U[0,1)^d, half-widths U[0.05,0.25), clipped to the cube; boxes
    containing init*1 or goal*1 are resampled."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    while len(out) < M:
        c = rng.random(d)
        hw = 0.05 + 0.2 * rng.random(d)
        lo, hi = np.clip(c - hw, 0, 1), np.clip(c + hw, 0, 1)
        if np.all((lo <= init) & (init <= hi)) or np.all((lo <= goal) & (goal <= hi)):
            continue
        out.append((lo, hi))
    return out
