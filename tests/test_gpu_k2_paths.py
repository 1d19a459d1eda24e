"""Every branch of the d = 2, 3 grid r-ball build (K1 grid + K2 count / fill: csrc/grid_rball.cu) against the
brute-force oracle: the one-round (<= 32 entries) and two-round (33..64) register fill, the warp path of rball_fill_big
for long columns and for columns with more than 255 candidates, its shared-memory rank sort (<= 256 entries) and the
spill + sort_big_columns path, the capped and the one-cell grid, flat sets, cell-face points, shards over unsorted and
x-sorted samples, rebuilds on one device table (speculative fill used, skipped on the device and relaunched), the
MPB200_FILL_U / MPB200_NO_GRAPH / MPB200_NO_SPEC_FILL switches and the N < 2^26 key-packing limit.  Sets and distances
must be byte-equal to the oracle.

Each case also asserts that its input reaches the branch it is named for, through k2_path(): a plain-Python copy of the
host geometry of build_table<D> and of the per-column dispatch of rball_count / rball_fill / rball_fill_big, evaluated
with the reference table's hit counts.  The copy is checked without a GPU on hand-worked cases (test_k2_geometry_*) and
on every case's input (test_k2_dispatch_replica)."""
import functools
import gc
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRID_SRC = os.path.join(ROOT, "motionplanning.jl_b200", "csrc", "grid_rball.cu")

MAX_PER_DIM = {2: 4096, 3: 256}
LIST_CAP = 64          # kListCap: hits of a register-filled column
MAX_CAND = 255         # kMaxCand: candidates addressable by the one-byte hit list
STAGE_CAP = 256        # kStageCap: hits rank-sorted in shared memory by rball_fill_big
KEY_LIMIT = 1 << 26    # the fill packs index << 6 | slot into 32 bits: N < 2^26
BRANCHES = ("empty", "one", "two", "stage", "spill")


# ---- plain-Python copy of the host geometry (build_table<D>) and of the per-column dispatch -------------------------
def grid_geometry(V, r, q0, q1):
    """bb = the query shard's box grown by r (clipped to the samples' box), the cell edge h (capped at 4096 / 256 cells
    per dimension), cells per dimension n, and the insertion box [in_lo, in_hi] = bb"""
    N, D = V.shape
    blo = [float(x) for x in V.min(axis=0)]
    bhi = [float(x) for x in V.max(axis=0)]
    if q1 > q0 and (q0, q1) != (0, N):
        qlo = [float(x) for x in V[q0:q1].min(axis=0)]
        qhi = [float(x) for x in V[q0:q1].max(axis=0)]
    else:
        qlo, qhi = blo, bhi
    grow = r * (1.0 + 1e-6)
    lo, hi = [], []
    for i in range(D):
        pad = grow + 4.5e-16 * max(abs(qlo[i]), abs(qhi[i]))
        a, b = max(blo[i], qlo[i] - pad), min(bhi[i], qhi[i] + pad)
        if not a <= b:
            a = b = blo[i]
        lo.append(a)
        hi.append(b)
    mpd = MAX_PER_DIM[D]
    ext_max = 0.0
    for i in range(D):
        ext_max = max(ext_max, hi[i] - lo[i])
    h = r * (1.0 + 1e-6)
    capped = not h > ext_max / mpd
    if capped:
        h = ext_max / mpd
    if not h > 0:
        h = 1.0
    n = tuple(int(min(np.floor((hi[i] - lo[i]) / h) + 1.0, mpd + 1)) for i in range(D))
    return dict(lo=tuple(lo), hi=tuple(hi), h=h, inv_h=1.0 / h, n=n, h_capped=capped)


def cell_of(g, P):
    """floor((p - lo) * inv_h), clamped to the grid: numpy rounds each operation like __dsub_rn / __dmul_rn"""
    c = np.empty(P.shape, dtype=np.int64)
    for i in range(P.shape[1]):
        q = np.floor((P[:, i] - g["lo"][i]) * g["inv_h"])
        c[:, i] = np.clip(q, 0, g["n"][i] - 1)
    return c


def k2_path(V, r, q0, q1, ref):
    """The branches build_table<D> takes for query columns [q0, q1), from the reference table of those columns
    (ref[0] = colptr as the oracle returns it)."""
    V = np.ascontiguousarray(V, dtype=np.float64)
    N, D = V.shape
    g = grid_geometry(V, r, q0, q1)
    inserted = np.ones(N, dtype=bool)
    for i in range(D):
        inserted &= (V[:, i] >= g["lo"][i]) & (V[:, i] <= g["hi"][i])
    n = g["n"]
    c = cell_of(g, V)
    lin = np.zeros(N, dtype=np.int64)
    for i in range(D - 1, -1, -1):
        lin = lin * n[i] + c[:, i]
    hist = np.bincount(lin[inserted], minlength=int(np.prod(n))).reshape(n[::-1])
    # candidates of a query: the samples in its 3 (d = 2) or 9 (d = 3) x-runs = the 3^d cells around its cell, clipped
    P = np.pad(hist, 1)
    box = np.zeros_like(hist)
    for off in np.ndindex(*(3,) * D):
        box += P[tuple(slice(o, o + m) for o, m in zip(off, hist.shape))]
    cq = c[q0:q1]
    total = box[tuple(cq[:, i] for i in range(D - 1, -1, -1))]
    cnt = np.diff(np.asarray(ref[0], dtype=np.int64))
    list_cap = LIST_CAP if N < KEY_LIMIT else 0
    big = (cnt > 0) & ((cnt > list_cap) | (total > MAX_CAND))
    cols = {"empty": cnt == 0,
            "one": ~big & (cnt > 0) & (cnt <= 32),
            "two": ~big & (cnt > 32),
            "stage": big & (cnt <= STAGE_CAP),
            "spill": big & (cnt > STAGE_CAP)}
    g.update(cnt=cnt, total=total, cols=cols, list_cap=list_cap, n_big=int(big.sum()), inserted=inserted,
             sorted_x=bool(N < 2 or np.all(V[:-1, 0] <= V[1:, 0])),
             empty_many=int((cols["empty"] & (total > MAX_CAND)).sum()))
    return g


def lengths(path, branch):
    return set(path["cnt"][path["cols"][branch]].tolist())


# ---- references ------------------------------------------------------------------------------------------------------
def np_rball(V, r, q0=0, q1=None):
    """the reference's operation order, one rounding per numpy operation (no FMA): s = (a0-b0)^2, s += (ai-bi)^2,
    member iff j != v and s <= r*r, value sqrt(s), rows ascending"""
    V = np.ascontiguousarray(V, dtype=np.float64)
    N, D = V.shape
    q1 = N if q1 is None else q1
    r2 = r * r
    colptr, rows, vals = [np.ones(1, dtype=np.int64)], [], []
    for a in range(q0, q1, 256):
        b = min(a + 256, q1)
        t = V[a:b, None, 0] - V[None, :, 0]
        s = t * t
        for i in range(1, D):
            t = V[a:b, None, i] - V[None, :, i]
            s = s + t * t
        m = s <= r2
        m[np.arange(b - a), np.arange(a, b)] = False
        qi, j = np.nonzero(m)
        rows.append(j.astype(np.int64) + 1)
        vals.append(np.sqrt(s[qi, j]))
        colptr.append(np.bincount(qi, minlength=b - a).astype(np.int64))
    cp = np.cumsum(np.concatenate(colptr))
    return cp, np.concatenate(rows) if rows else np.zeros(0, np.int64), np.concatenate(vals) if vals else np.zeros(0)


def _assert_same(got, ref, what):
    assert np.array_equal(got[0], ref[0]), "%s: colptr" % what
    assert np.array_equal(got[1], ref[1]), "%s: rowval" % what
    assert np.ascontiguousarray(got[2]).tobytes() == np.ascontiguousarray(ref[2]).tobytes(), "%s: nzval" % what


def _reference(orc, V, r, q0=0, q1=None):
    """oracle table; sets up to ~20k samples are also checked against the numpy restatement"""
    ref = orc.rball_brute(V, r, 0, q0, len(V) if q1 is None else q1)
    if len(V) <= 24000:
        _assert_same(np_rball(V, r, q0, q1), ref, "numpy restatement vs oracle")
    return ref


# ---- inputs ----------------------------------------------------------------------------------------------------------
SNAP = 2.0 ** -20      # coordinates on this lattice: offsets of k * 2^-8 are exact, and so are the distances below
# integer offsets (in units of u) at exactly 5 u (d = 2) or 13 u (d = 3): members exactly at the radius r = 5 u / 13 u
EXACT = {2: (5, np.array([[3, 4], [5, 0], [0, -5], [-4, -3]], dtype=np.float64)),
         3: (13, np.array([[3, 4, 12], [5, 12, 0], [-12, 0, -5], [0, -13, 0]], dtype=np.float64))}


def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def _snap(P):
    return np.round(np.asarray(P) / SNAP) * SNAP


def _exact_partners(rng, P, d, u, k):
    """for k of the points P, a partner at one of the EXACT offsets (scaled by u): exactly at distance EXACT[d][0] * u"""
    pick = rng.choice(len(P), size=min(k, len(P)), replace=False)
    return P[pick] + EXACT[d][1][rng.integers(0, len(EXACT[d][1]), size=len(pick))] * u


def _uniform(rng, n, d, avoid=(), clear=0.0):
    """n snapped uniform points of [0, 1)^d, none within Chebyshev distance `clear` of a point of `avoid`"""
    out = np.empty((0, d))
    avoid = np.asarray(avoid, dtype=np.float64).reshape(-1, d)
    while len(out) < n:
        P = _snap(rng.random((2 * n, d)))
        if len(avoid):
            P = P[(np.abs(P[:, None, :] - avoid[None, :, :]).max(-1) > clear).all(1)]
        out = np.vstack([out, P])
    return out[:n]


def _clique(rng, k, centre, r):
    """k snapped points within 0.45 r of centre: all pairwise within r"""
    d = len(centre)
    return _snap(np.asarray(centre) + (rng.random((k, d)) - 0.5) * (0.9 * r / np.sqrt(d)))


R = {2: 5 * 2.0 ** -8, 3: 13 * 2.0 ** -8}   # the EXACT radii with u = 2^-8
STAR_SIZES = (32, 33, 64, 65, 256, 257)
STAR_CENTRES = {2: [(0.2, 0.25), (0.5, 0.25), (0.8, 0.25), (0.2, 0.7), (0.5, 0.7), (0.8, 0.7)],
                3: [(0.25, 0.25, 0.25), (0.75, 0.25, 0.25), (0.25, 0.75, 0.25), (0.75, 0.75, 0.25),
                    (0.25, 0.25, 0.75), (0.75, 0.25, 0.75)]}


def case_lengths(d):
    """cliques of 33, 34, 65, 66, 257 and 258 samples in clearings of a uniform background: every sample of a clique
    has a column of exactly 32, 33, 64, 65, 256 or 257 entries and at most 258 candidates.  The background has
    partners exactly at r."""
    rng = _rng(5100 + d)
    r = R[d]
    centres = _snap(STAR_CENTRES[d])
    bg = _uniform(rng, 10000 if d == 2 else 16000, d, centres, 3.5 * r)
    parts = [bg, _exact_partners(rng, bg, d, 2.0 ** -8, 300)]
    parts[1] = parts[1][(np.abs(parts[1][:, None, :] - centres[None]).max(-1) > 2.5 * r).all(1)]
    for k, c in zip(STAR_SIZES, centres):
        parts.append(_clique(rng, k, c, r))
        parts.append(c[None, :])
    V = np.vstack(parts)
    return V[_rng(5150 + d).permutation(len(V))], r


def case_totals(d):
    """three queries in clearings, each with 3 partners exactly at r and dense clumps in the cells around it, every clump
    sample farther than r from it: 255 candidates (register fill), 256 candidates (rball_fill_big) and 0 hits with 301
    candidates (not filled).  The corners of the unit cube fix the grid: lo = 0, h = r (1 + 1e-6)."""
    rng = _rng(5200 + d)
    u = 2.0 ** -8
    r = 5 * u
    h = r * (1.0 + 1e-6)
    spots = [(0.25,) * d, (0.5,) * d, (0.75,) * d]
    corners = np.array(list(np.ndindex(*(2,) * d)), dtype=np.float64)
    bg = _uniform(rng, 6000 if d == 2 else 20000, d, spots, 5.5 * h)
    away = {2: np.array([[0, 5], [-4, -3], [-5, 0]], dtype=np.float64),             # partners away from the clumps
            3: np.array([[-3, -4, 0], [0, -3, -4], [-5, 0, 0]], dtype=np.float64)}[d] * u
    # clump cell offsets (one x-run each); in a cell at offset +1 / -1 / 0 a clump fills [1.6, 1.9] / [-0.9, -0.6] /
    # [0.3, 0.7] cell edges from the query's cell corner: at least 1.1 h from the query, which sits at the cell centre
    clump_cells = {2: [(1, 0), (-1, 1)], 3: [(1, 0, 0), (-1, 1, 0), (0, -1, 1)]}[d]
    span = {1: (1.6, 1.9), -1: (-0.9, -0.6), 0: (0.3, 0.7)}
    parts = [bg, corners]
    for spot, (partners, clump) in zip(spots, ((3, 251), (3, 252), (0, 300))):
        cell = np.floor(np.asarray(spot) / h)
        q = _snap((cell + 0.5) * h)
        parts += [q[None, :], q + away[:partners]]
        sizes = [clump // len(clump_cells)] * len(clump_cells)
        sizes[0] += clump - sum(sizes)
        for off, m in zip(clump_cells, sizes):
            a = np.array([(cell[i] + span[off[i]][0]) * h for i in range(d)])
            b = np.array([(cell[i] + span[off[i]][1]) * h for i in range(d)])
            parts.append(_snap(a + rng.random((m, d)) * (b - a)))
    V = np.vstack(parts)
    return V[_rng(5250 + d).permutation(len(V))], r


def case_cap(d):
    """r far below extent / 4096 (d = 2) or extent / 256 (d = 3): the cell edge is the cap, not r; micro-pairs exactly
    at r"""
    rng = _rng(5300 + d)
    u = 2.0 ** -16 if d == 2 else 2.0 ** -12
    r = EXACT[d][0] * u
    bg = _uniform(rng, 20000, d)
    corners = np.array([(0.0,) * d, (1.0,) * d])
    return np.vstack([bg, _exact_partners(rng, bg, d, u, 4000), corners]), r


def case_one_cell(d, n):
    """r >= the extent: one cell per dimension.  n = 64: every column is in the register fill (corners exactly 1 apart
    at r = 1); n = 300 at r = 2: all pairs, every column spilled"""
    rng = _rng(5400 + d + n)
    corners = np.array(list(np.ndindex(*(2,) * d)), dtype=np.float64)
    V = np.vstack([_snap(rng.random((n - len(corners), d))), corners])
    return V[rng.permutation(len(V))], (1.0 if n == 64 else 2.0)


def case_flat(d, kind):
    """extent 0 in one dimension (on a line in d = 2, on a plane in d = 3) or two (on a line in d = 3)"""
    rng = _rng(5500 + d + len(kind))
    n = {"line": 1500, "plane": 8000}[kind]
    free = 1 if kind == "line" else 2
    V = np.full((n, d), 0.375)
    V[:, :free] = _snap(rng.random((n, free)))
    V[n // 2:, 0] = V[:n // 2, 0] + 0.75 * R[2] * (rng.random(n - n // 2) < 0.5)   # some partners exactly 0.75 r apart
    return V, (R[2] if kind == "line" else 0.03)


def case_faces(d):
    """a dense block of the lattice 2^-13 Z^2 (2^-9 Z^3) with r = the spacing and the unit box: the capped cell edge is
    2^-12 (2^-8), so every other lattice point lies exactly on a cell face; axis neighbours are exactly at r"""
    s = 2.0 ** -13 if d == 2 else 2.0 ** -9
    rng_lo, k = (2001, 100) if d == 2 else (101, 22)
    idx = np.array(list(np.ndindex(*(k,) * d)), dtype=np.float64) + rng_lo
    V = np.vstack([idx * s, [(0.0,) * d, (1.0,) * d]])
    return V[_rng(5600 + d).permutation(len(V))], s


def case_negative(d):
    V, r = case_lengths(d)
    return V - (3.0 if d == 2 else 7.0), r             # exact: the snapped coordinates keep 22 bits


def case_offset(d):
    """a small cloud at 1e6 + [0, 1)^d (exact: 40 significant bits); the 4.5e-16 |x| term of the padding is 4.5e-10"""
    rng = _rng(5700 + d)
    u = 2.0 ** -6 if d == 2 else 2.0 ** -7
    r = EXACT[d][0] * u
    bg = _snap(rng.random((2000 if d == 2 else 6000, d)))
    return np.vstack([bg, _exact_partners(rng, bg, d, u, 300)]) + 1e6, r


def lattice_sorted(d):
    """the x-sorted lattice 2^-6 {0..47} x {0..199} (2^-5 {0..11} x {0..19}^2): runs of 200 (400) equal x; r = two
    spacings (axis partners exactly at r)"""
    s = 2.0 ** -6 if d == 2 else 2.0 ** -5
    shape = (48, 200) if d == 2 else (12, 20, 20)
    V = np.array(list(np.ndindex(*shape)), dtype=np.float64) * s            # x outermost: sorted along x
    return V, 2 * s, shape


def case_lattice_shards(d):
    """lattice_sorted with samples added exactly on the middle shard's in_lo / in_hi, and shard bounds inside runs of
    equal x; returns V, r and the shard bounds [0, a), [a, b), [b, N)"""
    V, r, shape = lattice_sorted(d)
    run = int(np.prod(shape[1:]))
    a, b = 6 * run + 34, (shape[0] * 3 // 5) * run + 155
    g = grid_geometry(V, r, a, b)
    ys = V[:run, 1:][::7]
    on_lo = np.hstack([np.full((len(ys), 1), g["lo"][0]), ys])
    on_hi = np.hstack([np.full((len(ys), 1), g["hi"][0]), ys])
    W = np.vstack([V, on_lo, on_hi])
    order = np.argsort(W[:, 0], kind="stable")
    W = W[order]
    shift = int((on_lo[0, 0] < V[a:b, 0].min()) * len(on_lo))
    return W, r, a + shift, b + shift


def case_rebuild(d):
    """uniform background with a 100-sample clique (big columns) and exact-r partners; r2 = 1.7 r1 (d = 2) / 1.45 r1
    (d = 3) more than doubles nnz"""
    rng = _rng(5800 + d)
    r1 = 0.018 if d == 2 else 0.06
    bg = _uniform(rng, 12000, d)
    V = np.vstack([bg, _exact_partners(rng, bg, d, r1 / EXACT[d][0], 500), _clique(rng, 100, (0.5,) * d, r1)])
    return V, r1, r1 * (1.7 if d == 2 else 1.45)


CASES = {}
for _d in (2, 3):
    # column lengths 32 | 33 and 64 | 65 (register fill: one round | two rounds | warp path), 256 | 257 (stage | spill)
    CASES["lengths-d%d" % _d] = (lambda d=_d: case_lengths(d) + (0, None),
                                 dict(lengths={"one": {32}, "two": {33, 64}, "stage": {65, 256}, "spill": {257}}))
    # candidate totals 255 | 256 with 3 hits, and 0 hits with 301 candidates (not big, not filled)
    CASES["totals-d%d" % _d] = (lambda d=_d: case_totals(d) + (0, None),
                                dict(has={"one", "stage", "empty"}, pairs={("one", 3, 255), ("stage", 3, 256), ("empty", 0, 301)},
                                     empty_many=True))
    CASES["grid-cap-d%d" % _d] = (lambda d=_d: case_cap(d) + (0, None), dict(h_capped=True, has={"one"}))
    CASES["grid-one-cell-d%d" % _d] = (lambda d=_d: case_one_cell(d, 64) + (0, None),
                                       dict(n=(1,) * _d, has={"two"}, n_big=0))
    CASES["grid-one-cell-all-pairs-d%d" % _d] = (lambda d=_d: case_one_cell(d, 300) + (0, None),
                                                 dict(n=(1,) * _d, only={"spill"}))
    CASES["grid-faces-d%d" % _d] = (lambda d=_d: case_faces(d) + (0, None),
                                    dict(h_capped=True, faces=True, has={"one"}))
    CASES["grid-negative-d%d" % _d] = (lambda d=_d: case_negative(d) + (0, None),
                                       dict(lengths={"one": {32}, "two": {33, 64}, "stage": {65, 256}, "spill": {257}}))
    CASES["grid-offset1e6-d%d" % _d] = (lambda d=_d: case_offset(d) + (0, None), dict(has={"one", "two"}))
    # shards over an unsorted set (whole sample array looked at) and its x-sorted copy (stripe_range)
    CASES["shard-unsorted-d%d" % _d] = (lambda d=_d: case_lengths(d) + (1500, 4500),
                                        dict(sorted_x=False, has={"one", "two", "stage", "spill"}))
    CASES["shard-sorted-d%d" % _d] = (
        lambda d=_d: (lambda V, r: (V[np.argsort(V[:, 0], kind="stable")], r, 1500, 4500))(*case_lengths(d)),
        dict(sorted_x=True, has={"one", "stage"}))
    CASES["shard-lattice-runs-d%d" % _d] = (lambda d=_d: case_lattice_shards(d), dict(sorted_x=True, on_bounds=True))
CASES["grid-flat-line-d2"] = (lambda: case_flat(2, "line") + (0, None), dict(n1=1, has={"one", "two", "stage"}))
CASES["grid-flat-plane-d3"] = (lambda: case_flat(3, "plane") + (0, None), dict(n2=1, has={"one"}))
CASES["grid-flat-line-d3"] = (lambda: case_flat(3, "line") + (0, None), dict(n1=1, n2=1, has={"one", "two", "stage"}))


def _check_path(name, V, r, q0, q1, ref, expect=None):
    path = k2_path(V, r, q0, q1, ref)
    e = CASES[name][1] if expect is None else expect
    for branch, want in e.get("lengths", {}).items():
        assert want <= lengths(path, branch), (name, branch, sorted(lengths(path, branch))[-8:])
    for branch in e.get("has", ()):
        assert path["cols"][branch].any(), (name, branch)
    if "only" in e:
        assert {b for b in BRANCHES if path["cols"][b].any()} == e["only"], name
    for branch, k, t in e.get("pairs", ()):
        sel = path["cols"][branch] & (path["cnt"] == k) & (path["total"] == t)
        assert sel.any(), (name, branch, k, t)
    if e.get("empty_many"):
        assert path["empty_many"] > 0, name
    if "h_capped" in e:
        assert path["h_capped"] == e["h_capped"], (name, path["h"])
    if "n" in e:
        assert path["n"] == e["n"], (name, path["n"])
    for i, key in ((1, "n1"), (2, "n2")):
        if key in e:
            assert path["n"][i] == e[key], (name, path["n"])
    if "n_big" in e:
        assert path["n_big"] == e["n_big"], name
    if "sorted_x" in e:
        assert path["sorted_x"] == e["sorted_x"], name
    if e.get("faces"):
        on_face = np.zeros(len(V), dtype=bool)
        for i in range(V.shape[1]):
            q = (V[:, i] - path["lo"][i]) * path["inv_h"]
            on_face |= (q == np.floor(q)) & (q > 0)
        assert on_face.sum() > len(V) // 3, name
    if e.get("on_bounds"):
        x = V[:, 0]
        assert (x == path["lo"][0]).any() and (x == path["hi"][0]).any(), name
        assert path["inserted"][(x == path["lo"][0]) | (x == path["hi"][0])].all(), name
        assert x[q0 - 1] == x[q0] and x[q1 - 1] == x[q1], name                      # shard bounds inside runs
    return path


# ---- the dispatch copy, without a GPU --------------------------------------------------------------------------------
def test_k2_geometry_cell_face_and_cap():
    """unit box, r = 2^-14 < 1/4096: h = 2^-12 exactly (the cap), 4097 cells; a point on the face x = 1/2 is in cell
    2048, one ulp below it in cell 2047, the top corner in the last cell"""
    V = np.array([[0.0, 0.0], [1.0, 1.0], [0.5, 0.25], [0.5 - 2.0 ** -54, 0.25 + 2.0 ** -12]])
    g = grid_geometry(V, 2.0 ** -14, 0, 4)
    assert g["h_capped"] and g["h"] == 2.0 ** -12 and g["inv_h"] == 4096.0 and g["n"] == (4097, 4097)
    assert g["lo"] == (0.0, 0.0) and g["hi"] == (1.0, 1.0)
    assert cell_of(g, V).tolist() == [[0, 0], [4096, 4096], [2048, 1024], [2047, 1025]]
    # not capped: r = 0.1, 1 / h = 9.99999.. -> 10 cells; 3-D cap: r = 1e-3 < 1/256 -> h = 1/256, 257 cells
    g = grid_geometry(np.array([[0.0, 0.0], [1.0, 0.5]]), 0.1, 0, 2)
    assert not g["h_capped"] and g["h"] == 0.1 * (1.0 + 1e-6) and g["n"] == (10, 5)
    g = grid_geometry(np.array([[0.0, 0.0, 0.0], [1.0, 1.0, 0.0]]), 1e-3, 0, 2)
    assert g["h_capped"] and g["h"] == 1.0 / 256 and g["n"] == (257, 257, 1)


def test_k2_geometry_shard_box():
    """shard [2, 4) of x in {0, 1, 2, 3, 10}: its box [2, 3] x [0.5, 1.5] grown by r (1 + 1e-6) + 4.5e-16 max|.|; in y
    both ends are clipped to the samples' box [0, 2]"""
    V = np.array([[0.0, 0.0], [1.0, 1.0], [2.0, 0.5], [3.0, 1.5], [10.0, 2.0]])
    g = grid_geometry(V, 0.5, 2, 4)
    pad_x = 0.5 * (1.0 + 1e-6) + 4.5e-16 * 3.0
    assert g["lo"] == (2.0 - pad_x, 0.0) and g["hi"] == (3.0 + pad_x, 2.0)
    assert g["n"] == (int(np.floor((g["hi"][0] - g["lo"][0]) / g["h"])) + 1, 4)
    p = k2_path(V, 0.5, 2, 4, (np.array([1, 1, 1]),))
    assert p["inserted"].tolist() == [False, False, True, True, False]
    # the full range: the samples' own box
    assert grid_geometry(V, 0.5, 0, 5)["lo"] == (0.0, 0.0)


def test_k2_geometry_candidate_totals():
    """a query at a cell centre, m samples in the next cell beyond r, none within r: total = m + 1.  With 3 hits, 255
    candidates is the register fill and 256 is big; without hits a column is never big; 64 hits is the two-round
    register fill and 65 goes to the warp path"""
    h = 1.0 * (1.0 + 1e-6)
    q = np.array([[2.5 * h, 2.5 * h]])
    corners = np.array([[0.0, 0.0], [8.0, 8.0]])

    def query(V, hits):                               # the full-range build, the query's column alone has entries
        cnt = np.zeros(len(V), dtype=np.int64)
        cnt[0] = hits
        p = k2_path(V, 1.0, 0, len(V), (np.concatenate([[1], 1 + np.cumsum(cnt)]),))
        assert p["n"] == (8, 8)
        return p, {b for b in BRANCHES if p["cols"][b][0]}

    for m in (254, 255):
        clump = np.column_stack([np.full(m, 3.8 * h), np.linspace(2.2, 2.8, m) * h])
        V = np.vstack([q, clump, corners])
        p, branch = query(V, 0)
        assert p["total"][0] == m + 1 and branch == {"empty"} and p["n_big"] == 0 and (p["empty_many"] > 0) == (m == 255)
        p, branch = query(V, 3)
        assert branch == {"one" if m == 254 else "stage"} and p["n_big"] == (m == 255)
    V = np.vstack([q, corners])
    assert query(V, 64)[1] == {"two"} and query(V, 65)[1] == {"stage"} and query(V, 257)[1] == {"spill"}


def test_k2_key_packing_limit_arithmetic():
    """the 8192 x 8192 lattice of the key-limit case: a 4097 x 4097 capped grid, at most 49 candidates per query, and the
    largest real key of N = 2^26 - 1 samples is 0xffffffbf, below the sentinel; one more sample would reach it"""
    s = 2.0 ** -13
    g = grid_geometry(np.array([[0.0, 0.0], [8191 * s, 8191 * s]]), 1.2 * s, 0, 2)
    assert g["h_capped"] and g["n"] == (4097, 4097)
    cx = cell_of(g, np.column_stack([np.arange(8192) * s, np.zeros(8192)]))[:, 0]
    per_cell = np.bincount(cx, minlength=4097)
    box = np.convolve(per_cell, np.ones(3, dtype=np.int64), mode="same")
    assert box.max() ** 2 <= 49                       # the 3 x 3 cells around a query hold at most 7 x 7 samples
    top = (KEY_LIMIT - 2) << 6 | 63
    assert top == 0xffffffbf and ((KEY_LIMIT - 1) << 6 | 63) == 0xffffffff


@pytest.mark.parametrize("name", list(CASES))
def test_k2_dispatch_replica(orc, name):
    """each case's input reaches the branch it is named for"""
    V, r, q0, q1 = CASES[name][0]()
    q1 = len(V) if q1 is None else q1
    _check_path(name, V, r, q0, q1, _reference(orc, V, r, q0, q1))


def test_k2_dispatch_replica_rebuild_and_switch_inputs(orc):
    """the rebuild input more than doubles nnz from r1 to r2 and has big columns; the switch sequence r, 1.25 r, r / 8
    over the lengths input has big columns in its first two builds and none in the third"""
    for d in (2, 3):
        V, r1, r2 = case_rebuild(d)
        ref1, ref2 = orc.rball_brute(V, r1), orc.rball_brute(V, r2)
        assert ref2[0][-1] - 1 > 2 * (ref1[0][-1] - 1)
        assert k2_path(V, r1, 0, len(V), ref1)["n_big"] > 0
        big = [p["n_big"] for p in _switch_input(orc, d)[3]]
        assert big[0] > 0 and big[1] > 0 and big[2] == 0, big


# ---- on the GPU --------------------------------------------------------------------------------------------------------
def _build(mp, V, r, q0=0, q1=None):
    NN = mp.MetricNN(V)
    q1 = len(V) if q1 is None else q1
    if (q0, q1) != (0, len(V)):
        NN.set_query_range(q0, q1)
    D = NN.precompute(r).D
    out = (np.array(D.colptr), np.array(D.rowval), np.array(D.nzval))
    NN.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_k2_path_matches_oracle(gpu, orc, name):
    V, r, q0, q1 = CASES[name][0]()
    q1 = len(V) if q1 is None else q1
    ref = _reference(orc, V, r, q0, q1)
    _check_path(name, V, r, q0, q1, ref)
    _assert_same(_build(gpu, V, r, q0, q1), ref, name)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 3])
def test_k2_shards_concatenate_to_the_full_build(gpu, orc, d):
    """shards [0, a), [a, b), [b, N) of the x-sorted lattice, bounds inside runs of equal x, the first shard's in_lo and
    the last shard's in_hi on the samples' box: each equals the oracle and their rows and values are the full build's"""
    V, r, a, b = case_lattice_shards(d)
    N = len(V)
    full_ref = _reference(orc, V, r)
    full = _build(gpu, V, r)
    _assert_same(full, full_ref, "full range")
    rows, vals = [], []
    for q0, q1 in ((0, a), (a, b), (b, N)):
        ref = _reference(orc, V, r, q0, q1)
        path = k2_path(V, r, q0, q1, ref)
        assert path["sorted_x"]
        if q0 == 0:
            assert path["lo"][0] == V[0, 0] and path["inserted"][V[:, 0] == path["lo"][0]].all()
        if q1 == N:
            assert path["hi"][0] == V[-1, 0] and path["inserted"][V[:, 0] == path["hi"][0]].all()
        got = _build(gpu, V, r, q0, q1)
        _assert_same(got, ref, "shard [%d, %d)" % (q0, q1))
        rows.append(got[1])
        vals.append(got[2])
    assert np.array_equal(np.concatenate(rows), full[1])
    assert np.concatenate(vals).tobytes() == full[2].tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 3])
def test_k2_rebuilds_on_one_table(gpu, orc, d):
    """one MetricNN and its one device table: fresh r1 (no speculative fill), r2 with nnz > capacity (the speculative
    fill returns on the device and the fill is launched again), r2 again (graph replayed, speculative fill used), r1
    again (speculative fill used, a stale tail past nnz), a shard and the full range again (graph captured again)"""
    from mpb200 import _lib
    lib = _lib.lib()
    V, r1, r2 = case_rebuild(d)
    N = len(V)
    q0, q1 = 3001, 9002
    refs = {r1: _reference(orc, V, r1), r2: _reference(orc, V, r2)}
    shard_ref = _reference(orc, V, r1, q0, q1)
    assert refs[r2][0][-1] - 1 > 2 * (refs[r1][0][-1] - 1)
    gc.collect()
    _lib.check(lib.mpb200_release_cached())               # no parked block larger than the r1 table is handed out
    NN = gpu.MetricNN(V)
    NN.handle()      # the sample set is created on first use; its bounding-box launches are not the build's

    def build(r, ref, what):
        before = lib.mpb200_launch_count()
        NN.build_table(r)
        launches = lib.mpb200_launch_count() - before
        D = NN.fetch_table(NN.table)
        _assert_same((np.array(D.colptr), np.array(D.rowval), np.array(D.nzval)), ref, what)
        return launches

    fresh = build(r1, refs[r1], "fresh r1")
    overflow = build(r2, refs[r2], "r2 over capacity")
    replay = build(r2, refs[r2], "r2 again")
    assert overflow - replay == 1                         # the speculative fill returned and was launched again
    assert build(r1, refs[r1], "r1 again") == fresh       # speculative fill in place of the plain one
    NN.set_query_range(q0, q1)
    build(r1, shard_ref, "shard")
    NN.set_query_range(0, N)
    build(r1, refs[r1], "full range again")
    NN.close()


def switch_radii(r):
    return (r, 1.25 * r, r / 8)


@functools.lru_cache(maxsize=None)
def _switch_input(orc, d):
    """the lengths input, its rebuild radii, their reference tables and paths (shared by the switch cases)"""
    V, r = case_lengths(d)
    radii = switch_radii(r)
    refs = [_reference(orc, V, rr) for rr in radii]
    return V, radii, refs, [k2_path(V, rr, 0, len(V), ref) for rr, ref in zip(radii, refs)]


def _launch_lines():
    """grid_rball.cu line numbers of the MPB_LAUNCHED() after the rball_fill, rball_fill_big and sort_big_columns
    launches (the lines MPB200_TRACE lists)"""
    src = open(GRID_SRC).read().split("\n")
    out = {}
    for key, pat in (("fill", "rball_fill<D, 2><<<"), ("big", "rball_fill_big<D><<<"), ("sort", "sort_big_columns<<<")):
        start = next(i for i, line in enumerate(src) if pat in line)
        out[key] = next(i for i in range(start, len(src)) if "MPB_LAUNCHED();" in src[i]) + 1
    return out


_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import mpb200
V = np.load(sys.argv[2])
radii = [float(x) for x in sys.argv[3].split(",")]
mpb200.init(0)
NN = mpb200.MetricNN(V)
out = []
for r in radii:                                 # one table, rebuilt
    D = NN.precompute(r).D
    out += [np.array(D.colptr), np.array(D.rowval), np.array(D.nzval)]
mpb200.load().mpb200_synchronize()              # with MPB200_TRACE set, the launches of all builds are listed here
np.savez(sys.argv[4], *out)
NN.close()
"""


@pytest.mark.gpu
@pytest.mark.parametrize("d", [2, 3])
@pytest.mark.parametrize("switch", ["MPB200_FILL_U=1", "MPB200_FILL_U=2", "MPB200_FILL_U=4", "MPB200_NO_GRAPH=1",
                                    "MPB200_NO_SPEC_FILL=1"])
def test_k2_switches_match_oracle(gpu, orc, tmp_path, switch, d):
    """the switches are read once per process: each sequence of builds runs in a child process of its own.  Its launch
    trace lists rball_fill_big and sort_big_columns exactly in the builds with big columns"""
    V, radii, refs, paths = _switch_input(orc, d)
    assert all(paths[0]["cols"][b].any() for b in ("one", "two", "stage", "spill"))
    np.save(tmp_path / "V.npy", V)
    key, val = switch.split("=")
    res = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path / "V.npy"), ",".join(map(repr, radii)),
                          str(tmp_path / "out.npz")],
                         env=dict(os.environ, MPB200_TRACE="1", **{key: val}), capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    got = np.load(tmp_path / "out.npz")
    for i, (rr, ref) in enumerate(zip(radii, refs)):
        _assert_same(tuple(got["arr_%d" % (3 * i + k)] for k in range(3)), ref, "%s build %d (r = %r)" % (switch, i, rr))
    # one trace segment per build, each starting at its phase mark 0
    lines = _launch_lines()
    trace = [ln for ln in res.stderr.splitlines() if ln.startswith("[trace]")]
    builds, cur = [], None
    for ln in trace:
        m = re.match(r"\[trace\]\s+(\S+?)\s*:(\d+)", ln)
        if m.group(1) == "phase" and m.group(2) == "0":
            cur = []
            builds.append(cur)
        elif cur is not None and m.group(1) == "grid_rball.cu":
            cur.append(int(m.group(2)))
    assert len(builds) == len(radii), res.stderr[-3000:]
    for i, (seg, path) in enumerate(zip(builds, paths)):
        assert (lines["big"] in seg) == (path["n_big"] > 0), (i, seg)
        assert (lines["sort"] in seg) == (path["n_big"] > 0), (i, seg)
        assert lines["fill"] in seg, (i, seg)
        if key == "MPB200_NO_SPEC_FILL":
            assert seg.count(lines["fill"]) == 1, (i, seg)


# ---- the N < 2^26 key-packing limit ------------------------------------------------------------------------------------
KEY_SIDE = 8192
KEY_S = 2.0 ** -13


def _key_lattice():
    """V[k] = (k % 8192, k // 8192) * 2^-13, all 2^26 points"""
    k = np.arange(KEY_SIDE * KEY_SIDE, dtype=np.int64)
    V = np.empty((len(k), 2))
    V[:, 0] = (k % KEY_SIDE) * KEY_S
    V[:, 1] = (k // KEY_SIDE) * KEY_S
    return V


def _key_expected_counts(N):
    k = np.arange(N, dtype=np.int64)
    i, j = k % KEY_SIDE, k // KEY_SIDE
    cnt = (i > 0).astype(np.int64) + (j > 0) + ((i < KEY_SIDE - 1) & (k + 1 < N)) + ((j < KEY_SIDE - 1) & (k + KEY_SIDE < N))
    colptr = np.empty(N + 1, dtype=np.int64)
    colptr[0] = 1
    np.cumsum(cnt, out=colptr[1:])
    colptr[1:] += 1
    return colptr


@pytest.mark.gpu
def test_k2_key_packing_limit(gpu, orc):
    """N = 2^26 - 1 (the lattice minus its last point): every column in the register fill, the top index at the top of
    the 26-bit key field.  N = 2^26: list_cap = 0, every column through rball_fill_big, neither the fill nor the
    speculation runs -- exactly one launch more than N = 2^26 - 1 (rball_fill_big + sort_big_columns in place of
    rball_fill).  Each column holds its 2..4 axis neighbours at exactly 2^-13; the table is checked on the device."""
    import torch
    from mpb200 import _lib, sharding
    lib = _lib.lib()
    V = _key_lattice()
    r = 1.2 * KEY_S
    launches = {}
    for N in (KEY_LIMIT - 1, KEY_LIMIT):
        W = V[:N]
        colptr = _key_expected_counts(N)
        path = k2_path(W, r, 0, N, (colptr,))
        assert path["n"] == (4097, 4097) and path["h_capped"] and path["total"].max() <= 49
        if N < KEY_LIMIT:
            assert path["list_cap"] == LIST_CAP and path["n_big"] == 0 and path["cols"]["one"].all()
            assert ((N - 1) << 6 | 63) == 0xffffffbf
        else:
            assert path["list_cap"] == 0 and path["n_big"] == N and path["cols"]["stage"].all()
        del path
        gc.collect()
        _lib.check(lib.mpb200_release_cached())
        NN = gpu.MetricNN(W)
        NN.handle()  # the sample set is created on first use; its bounding-box launches are not the build's
        before = lib.mpb200_launch_count()
        NN.build_table(r)
        launches[N] = lib.mpb200_launch_count() - before
        _lib.check(lib.mpb200_synchronize())
        assert NN.table.nnz == colptr[-1] - 1
        cp, rv, nz, _ = sharding.table_device_tensors(NN.table)
        dev = cp.device
        k = torch.arange(N, dtype=torch.int64, device=dev)
        i, j = k % KEY_SIDE, k // KEY_SIDE
        cand = torch.stack([k - KEY_SIDE, k - 1, k + 1, k + KEY_SIDE], 1)
        ok = torch.stack([j > 0, i > 0, i < KEY_SIDE - 1, j < KEY_SIDE - 1], 1) & (cand < N)
        assert torch.equal(cp, torch.from_numpy(colptr).to(dev))
        del i, j, k
        assert torch.equal(rv, cand[ok] + 1)
        del cand, ok
        assert bool((nz == KEY_S).all())
        # windows against the oracle: the first and the last two rows; every neighbour of a column in them lies in the
        # rows next to them, so the oracle runs on that stretch of the lattice alone
        for c0, c1 in ((0, 2 * KEY_SIDE), (N - 2 * KEY_SIDE, N)):
            s0 = max(0, c0 - KEY_SIDE)
            s1 = min(N, c1 + KEY_SIDE)
            ref = orc.rball_brute(W[s0:s1], r, 0, c0 - s0, c1 - s0)
            got_cp = cp[c0:c1 + 1].cpu().numpy()
            a, b = int(got_cp[0]) - 1, int(got_cp[-1]) - 1
            got = (got_cp - got_cp[0] + 1, rv[a:b].cpu().numpy() - s0, nz[a:b].cpu().numpy())
            _assert_same(got, ref, "N = %d, columns [%d, %d)" % (N, c0, c1))
        del cp, rv, nz
        torch.cuda.synchronize()
        NN.close()
        NN.table.close()
        del NN
        gc.collect()
        torch.cuda.empty_cache()
        _lib.check(lib.mpb200_release_cached())
    assert launches[KEY_LIMIT] - launches[KEY_LIMIT - 1] == 1, launches
