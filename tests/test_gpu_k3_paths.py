"""Every branch of the d >= 4 Euclidean r-ball build (K3 + K4: csrc/brute_rball.cu dispatching into csrc/tc_rball.cu)
against the brute-force oracle: the symmetric tensor-core sweep and each of its slab merges, the one-sided sweep of
sharded builds and of full-range builds with a large slab, the count-only sweep feeding the CUDA-core fill, slab
overflow, every dimension 4..14 and the tile / padding edges.  Sets and distances must be byte-equal to the oracle.

Each case also asserts that its input reaches the branch it is named for, through k3_path(): a plain-Python copy of
the host dispatch of brute_build, evaluated on the reference table.  The copy is checked without a GPU
(test_k3_dispatch_replica); the tensor-core / CUDA-core choice is also witnessed on the GPU through MPB200_TRACE."""
import os
import subprocess
import sys

import numpy as np
import pytest

import fixtures as fx

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- plain-Python copy of the host dispatch (brute_rball.cu: brute_build, tc_rball.cu: tc_delta / tc_center) ----------
def tc_center(V):
    """centre of the samples' bounding box and the squared radius of the centred cloud"""
    lo, hi = V.min(axis=0), V.max(axis=0)
    center = 0.5 * (lo + hi)
    Rmax2 = 0.0
    for k in range(V.shape[1]):
        h = max(abs(lo[k] - center[k]), abs(hi[k] - center[k]))
        Rmax2 += h * h
    return center, float(Rmax2)


def tc_delta(r, Rmax2):
    u_tf32 = 4.8828125e-4
    e_dot = 2.0 * u_tf32 * (1.0 + u_tf32) * Rmax2
    e_acc = 64.0 * 1.1920929e-7 * (Rmax2 + 0.5 * (r * r + Rmax2))
    e_thr = 3.6e-7 * 0.5 * (r * r + Rmax2)
    return float(np.float32(1.5 * (e_dot + e_acc + 2.0 * e_thr) + 1e-30))


def band_ratio(V, r):
    """2 delta / r^2: the tensor-core prefilter is used while this is at most 0.25"""
    return 2.0 * tc_delta(r, tc_center(V)[1]) / (r * r)


def tc_band_is_tight(V, r):
    return 2.0 * tc_delta(r, tc_center(V)[1]) <= 0.25 * r * r


def k3_path(V, r, q0, q1, colptr, rowval, env=()):
    """The branches brute_build takes for query columns [q0, q1), from the reference table of those columns
    (colptr, rowval as the oracle returns them); env: the MPB200_* switches set in the building process.
    Assumes the slabs fit in device memory (otherwise the build takes the two-sweep fill from the start)."""
    N, d = V.shape
    nq = q1 - q0
    counts = np.diff(colptr)
    tc = 4 <= d <= 14 and "MPB200_NO_TC" not in env and tc_band_is_tight(V, r)
    cap = 0
    if nq > 0:
        probe = min(nq, 2048)
        h_max = int(counts[:probe].max())
        cap = h_max if probe == nq else h_max + h_max // 2 + 64
        cap = (cap + 31) & ~31
    single = cap > 0
    symmetric = single and tc and "MPB200_TC_FULL" not in env and nq == N and q0 == 0 and cap <= 8192
    sweep = "none" if nq == 0 else "symmetric" if symmetric else "one-sided" if single else "count"
    overflow = single and int(counts.max()) > cap
    fill, merges = None, set()
    if nq > 0 and colptr[-1] > colptr[0]:
        fill = "two-sweep" if (not single or overflow) else "merge" if symmetric else "slab"
    if fill == "merge":
        np_, slot_bits = 64, 6
        while np_ < cap:
            np_ <<= 1
            slot_bits += 1
        idx_bits = 1
        while (1 << idx_bits) < N:
            idx_bits += 1
        block = "block32" if idx_bits + slot_bits <= 32 else "block64"
        cols = np.repeat(np.arange(q0, q1, dtype=np.int64), counts)
        kr = np.bincount(cols[rowval - 1 < cols], minlength=nq)      # entries with a smaller index than the column
        if idx_bits <= 22 and "MPB200_SLAB_BLOCK_SORT" not in env:
            for lo, hi, name in ((1, 64, "warp2"), (65, 128, "warp4"), (129, 256, "warp8"), (257, 512, "warp16"),
                                 (513, 1024, "wide"), (1025, 1 << 30, block)):
                if ((kr >= lo) & (kr <= hi)).any():
                    merges.add(name)
        else:
            merges.add(block)
    return dict(tc=bool(tc), cap=cap, sweep=sweep, overflow=bool(overflow), fill=fill, merges=merges)


# ---- inputs ----------------------------------------------------------------------------------------------------------
def _rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def _ball(rng, n, center, r):
    """n points within r/2 of center: every pair is within r"""
    d = len(center)
    return np.asarray(center) + (rng.random((n, d)) - 0.5) * (r / np.sqrt(d))


def _away(rng, n, d, center, dist):
    """n uniform points of the unit cube at least dist from center"""
    out = np.empty((0, d))
    while len(out) < n:
        P = rng.random((n, d))
        out = np.vstack([out, P[((P - center) ** 2).sum(1) >= dist * dist]])
    return out[:n]


def _lattice_sites(rng, n, d, k, step):
    """n distinct points of {0, step, .., (k-1) step}^d: pairwise at least step apart"""
    idx = rng.choice(k ** d, size=n, replace=False)
    return ((idx[:, None] // k ** np.arange(d)) % k).astype(np.float64) * step


def _uniform(d, N, seed, degree=30):
    """unit-cube cloud with ~degree entries per column, some exact duplicates (distance 0)"""
    V = _rng(seed).random((N, d))
    if N >= 64:
        V[N - 10:] = V[10:20]
    probe = V[:min(N, 200)]
    s = ((probe[:, None, :] - V[None, :, :]) ** 2).sum(-1)
    r = float(np.sqrt(np.quantile(s, min(1.0, degree / N))))
    return V, max(r, 0.35)


def case_a(d, shard):
    V, r = _uniform(d, 2500, 4100 + d)
    return (V, r, 37, 2461) if shard else (V, r, 0, 2500)


def case_b(d, N):
    V = _rng(4200 + 7 * d + N).random((N, d))
    return V, (0.35 if d == 4 else 0.6), 0, N


def case_c_shards():
    V, r = _uniform(6, 4000, 4301)
    return V, r, 1811          # shards [0, a) and [a, a+1): exact cap; [a+1, N): estimated cap


def case_c_band(offset):
    """lattice cloud with partners planted exactly at the radius, one ulp-scale step beyond it and just inside"""
    rng = _rng(4302)
    d, step = 5, 1.0 / 32
    base = fx.lattice_cloud(rng, 700, d, step, 0.0, 0.65)
    r = 10.0 / 32                       # |(6,8,0,0,0)| = |(5,5,5,5,0)| = |(8,4,4,2,0)| = 10
    dirs = np.array([[6, 8, 0, 0, 0], [5, 5, 5, 5, 0], [8, 4, 4, 2, 0]], dtype=np.float64)
    at_r = [base + dirs[k] * step for k in range(3)]
    beyond = base + dirs[0] * step
    beyond[:, 4] += 2.0 ** -20          # s = r^2 + 2^-40: not a member, deep inside the TF32 band
    inside = base + dirs[1] * step
    inside[:, 0] -= 2.0 ** -20          # s just below r^2
    return np.vstack([base] + at_r + [beyond, inside]) + offset, r


TF32_A = 0.5 + 2.0 ** -12 - 2.0 ** -24      # rounds down to 0.5 in TF32: the largest relative error there is


def case_c_tf32(q0, q1):
    """d = 14, samples on the corners (+-TF32_A)^14 and partners moved inwards by (6, 8)/16 in two coordinates: exactly
    at r = 10/16.  The other 12 coordinates are equal and every one of them rounds down in TF32, so the tensor-core dot
    product falls short by ~ -2^-12 * 12, more than half of the error allowance delta (the tight case for it)"""
    rng = _rng(4303)
    d = 14
    X = (2.0 * _lattice_sites(rng, 700, d, 2, 1.0) - 1.0) * TF32_A
    Y = X.copy()
    Y[:, 0] -= np.sign(X[:, 0]) * (6.0 / 16)
    Y[:, 1] -= np.sign(X[:, 1]) * (8.0 / 16)
    V = np.vstack([X, Y])
    return V, 10.0 / 16, q0, (len(V) if q1 is None else q1)


def tf32_dot_error(X, Y):
    """what TF32 operands (cvt.rna of the centred FP32 coordinates) take off the exact dot products X_i . Y_i"""
    def tf32(a):
        b = a.astype(np.float32).view(np.uint32)
        return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32).astype(np.float64)
    return (tf32(X) * tf32(Y)).sum(1) - (X * Y).sum(1)


def case_d(shard):
    """a tight cloud, then (after index 2048 of the probe window) a dense cluster whose columns overflow the slab"""
    rng = _rng(4400)
    d, r = 5, 0.25
    c = np.full(d, 0.5)
    V = np.vstack([_away(rng, 3300, d, c, 2 * r), _ball(rng, 600, c, r), _away(rng, 300, d, c, 2 * r)])
    return (V, r, 1001, 4111) if shard else (V, r, 0, len(V))


def case_e(q0, q1):
    """isolated samples (pairwise more than r apart) at indices 0 .. 2099 and 2400 .. 2599, a cluster in between"""
    rng = _rng(4500)
    d, r = 8, 0.45
    sites = _lattice_sites(rng, 2300, d, 3, 0.5)          # pairwise >= 0.5 apart
    cluster = _ball(rng, 300, [0.25] * d, r)              # >= sqrt(8)/4 - r/2 from every site
    V = np.vstack([sites[:2100], cluster, sites[2100:]])
    return V, r, q0, (len(V) if q1 is None else q1)


def case_f():
    """about 5500 samples mutually within r in the probe window: cap > 8192, full range on the one-sided sweep"""
    rng = _rng(4600)
    d, r = 4, 0.3
    V = np.vstack([_ball(rng, 5500, [0.5] * d, r), rng.random((2500, d))])
    return V, r, 0, len(V)


def case_g():
    """one symmetric build through every merge: a cluster of 3000 at the front (kr = 0 .. 2999), then a warp whose
    query 5 (the hub) has 400 partners of larger index while its 31 warp-mates, on cube corners, have none"""
    rng = _rng(4700)
    d, r = 6, 0.3
    corners = _lattice_sites(rng, 31, d, 2, 1.0)
    hub = np.array([0.7] * d)
    bg = lambda n: 0.35 + 0.45 * rng.random((n, d))      # farther than r from every corner
    V = np.vstack([_ball(rng, 3000, [0.3] * d, r), bg(72), corners[:5], hub, corners[5:], bg(296), _ball(rng, 400, hub, r),
                   bg(1200)])
    return V, r, 0, len(V), 3072 + 5


G64_N, G64_C = (1 << 19) + 1, 3000


def case_g64():
    """N just above 2^19 (20 index bits) and a cluster of 3000 (cap > 4096: 13 slot bits): 64-bit merge keys.
    The rest sit on distinct sites of {0, 1, 2}^12, pairwise 1 > r apart and > r from the cluster: their columns
    are empty, so the reference is the cluster's own table."""
    rng = _rng(4800)
    d, r = 12, 0.9
    sites = _lattice_sites(rng, G64_N - G64_C, d, 3, 1.0)
    V = np.vstack([_ball(rng, G64_C, [0.5] * d, r), sites])
    return V, r, 0, G64_N


def _g64_reference(orc, V, r):
    cp, rv, nz = orc.rball_brute(V[:G64_C], r)
    return np.concatenate([cp, np.full(G64_N - G64_C, cp[-1], dtype=np.int64)]), rv, nz


SHARDED = {"tc": True, "sweep": "one-sided", "fill": "slab"}
SYMMETRIC = {"tc": True, "sweep": "symmetric", "fill": "merge"}
CASES = {}
for _d in range(4, 15):
    CASES["a-d%d-full" % _d] = (lambda d=_d: case_a(d, False), SYMMETRIC)
    CASES["a-d%d-shard" % _d] = (lambda d=_d: case_a(d, True), SHARDED)
for _d in (4, 7):
    for _N in (1, 2, 31, 63, 64, 65, 127, 128, 129, 2048, 2049):
        CASES["b-d%d-N%d" % (_d, _N)] = (lambda d=_d, N=_N: case_b(d, N),
                                         SYMMETRIC if _N >= 31 else {"tc": True, "sweep": "count"} if _N == 1 else {"tc": True})
for _off in (0.0, 1000.0, -3.0e4):
    CASES["c-band%g-exact" % _off] = (lambda o=_off: case_c_band(o) + (100, 1901), SHARDED)
    CASES["c-band%g-estimated" % _off] = (lambda o=_off: case_c_band(o) + (1901, 4200), SHARDED)
CASES["c-tf32-rounding-full"] = (lambda: case_c_tf32(0, None), SYMMETRIC)
CASES["c-tf32-rounding-shard"] = (lambda: case_c_tf32(100, 1301), SHARDED)
CASES["d-overflow-full"] = (lambda: case_d(False), {"tc": True, "sweep": "symmetric", "overflow": True, "fill": "two-sweep"})
CASES["d-overflow-shard"] = (lambda: case_d(True), {"tc": True, "sweep": "one-sided", "overflow": True, "fill": "two-sweep"})
# a probe without entries estimates cap = 64 when it does not cover the range: the cluster overflows that slab;
# when it does cover the range, cap = 0 and the count-only sweep decides colptr (every column empty)
CASES["e-empty-probe-full"] = (lambda: case_e(0, None), {"tc": True, "cap": 64, "sweep": "symmetric", "overflow": True,
                                                         "fill": "two-sweep"})
CASES["e-empty-probe-shard"] = (lambda: case_e(3, 2555), {"tc": True, "cap": 64, "sweep": "one-sided", "overflow": True,
                                                          "fill": "two-sweep"})
CASES["e-count-only-shard"] = (lambda: case_e(3, 2003), {"tc": True, "cap": 0, "sweep": "count", "fill": None})
CASES["f-large-cap-full"] = (case_f, SHARDED)
CASES["g-merges"] = (lambda: case_g()[:4], dict(SYMMETRIC, merges={"warp2", "warp4", "warp8", "warp16", "wide", "block32"}))
CASES["g-merges-64bit-keys"] = (case_g64, dict(SYMMETRIC, merges={"warp2", "warp4", "warp8", "warp16", "wide", "block64"}))
HEAVY = {"g-merges-64bit-keys"}


def _reference(orc, name, V, r, q0, q1):
    if name == "g-merges-64bit-keys":
        return _g64_reference(orc, V, r)
    return orc.rball_brute(V, r, 0, q0, q1)


def _check_path(name, V, r, q0, q1, ref, env=(), expect=None):
    path = k3_path(V, r, q0, q1, ref[0], ref[1], env)
    if path["tc"]:
        assert band_ratio(V, r) <= 0.1, (name, band_ratio(V, r))     # well clear of the 0.25 cut
    for key, want in (expect if expect is not None else CASES[name][1]).items():
        if key == "merges":
            assert want <= path[key], (name, path)
        else:
            assert path[key] == want, (name, key, path)
    return path


# ---- the dispatch copy, without a GPU --------------------------------------------------------------------------------
@pytest.mark.parametrize("name", [n for n in CASES if n not in HEAVY])
def test_k3_dispatch_replica(orc, name):
    """each case's input reaches the branch it is named for"""
    V, r, q0, q1 = CASES[name][0]()
    path = _check_path(name, V, r, q0, q1, _reference(orc, name, V, r, q0, q1))
    if name.startswith("f-"):
        assert path["cap"] > 8192 and q0 == 0 and q1 == len(V)
    if name.endswith("-estimated") or name.startswith("a-") and name.endswith("-shard"):
        assert q1 - q0 > 2048
    if name.endswith("-exact"):
        assert q1 - q0 <= 2048
    if name == "c-tf32-rounding-full":
        X, Y = V[:700], V[700:]
        center, Rmax2 = tc_center(V)
        delta = tc_delta(r, Rmax2)
        err = tf32_dot_error(X - center, Y - center)
        assert (((X - Y) ** 2).sum(1) == r * r).all()                  # members, exactly at the radius
        assert -delta < err.min() and err.max() < -delta / 2          # within the allowance, using more than half of it


def test_k3_dispatch_replica_heavy_cases(orc):
    """the 64-bit-key case (reference built from its cluster alone) and the hub column of the merge case"""
    V, r, q0, q1 = case_g64()
    assert (np.abs(V[G64_C:] - 0.5) >= 0.5).all() and (np.abs(V[:G64_C] - 0.5) <= r / 2).all()  # sites > r from the cluster
    _check_path("g-merges-64bit-keys", V, r, q0, q1, _g64_reference(orc, V, r))
    V, r, q0, q1, hub = case_g()
    cp, rv, _ = orc.rball_brute(V, r)
    w0 = hub & ~31
    later = [int(((rv[cp[j] - 1:cp[j + 1] - 1] - 1) > j).sum()) for j in range(w0, w0 + 32)]
    assert later[hub - w0] >= 400 and sum(later) == later[hub - w0]


def test_k3_dispatch_replica_sends_the_wide_band_tests_to_the_cuda_cores(orc):
    """the inputs of test_k3_prefilter_band_has_no_false_negatives and test_k3_single_sweep_slab_overflow_falls_back
    (test_gpu_parity.py) take the FP32 CUDA-core prefilter, not the tensor cores"""
    rng = _rng(17)
    d = 5
    base = rng.integers(-40, 40, size=(600, d)).astype(np.float64)
    V = np.vstack([base, base + [3, 4, 0, 0, 0], base + [0, 0, 5, 0, 0], base + [3, 0, 4, 0, 1e-9]]) / 8.0
    for off, r in ((0.0, 5.0 / 8.0), (1000.0, 5.0 / 8.0), (-3.0e4, 0.7)):
        W = V + off
        ref = orc.rball_brute(W, r, 0, 100, 1900)
        assert k3_path(W, r, 100, 1900, ref[0], ref[1])["tc"] is False
    rng = _rng(5)
    V = np.vstack([rng.random((3000, d)), 3.0 + 0.01 * rng.random((700, d)), rng.random((300, d))])
    ref = orc.rball_brute(V, 0.12)
    path = k3_path(V, 0.12, 0, len(V), ref[0], ref[1])
    assert path["tc"] is False and path["overflow"] and path["fill"] == "two-sweep"
    # and MPB200_NO_TC takes every case to the CUDA cores
    V, r, q0, q1 = case_a(6, False)
    ref = orc.rball_brute(V, r)
    assert k3_path(V, r, q0, q1, ref[0], ref[1], {"MPB200_NO_TC"})["tc"] is False


# ---- on the GPU --------------------------------------------------------------------------------------------------------
def _build(mp, V, r, q0, q1):
    NN = mp.MetricNN(V)
    if (q0, q1) != (0, len(V)):
        NN.set_query_range(q0, q1)
    D = NN.precompute(r).D
    out = (np.array(D.colptr), np.array(D.rowval), np.array(D.nzval))
    NN.close()
    return out


def _assert_same(got, ref, what):
    assert np.array_equal(got[0], ref[0]), "%s: colptr" % what
    assert np.array_equal(got[1], ref[1]), "%s: rowval" % what
    assert got[2].tobytes() == np.ascontiguousarray(ref[2]).tobytes(), "%s: nzval" % what


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_k3_path_matches_oracle(gpu, orc, name):
    V, r, q0, q1 = CASES[name][0]()
    ref = _reference(orc, name, V, r, q0, q1)
    _check_path(name, V, r, q0, q1, ref)
    _assert_same(_build(gpu, V, r, q0, q1), ref, name)


@pytest.mark.gpu
def test_k3_tensor_core_shards_concatenate_to_the_symmetric_build(gpu, orc):
    """shards [0, a), [a, a+1), [a+1, N) with a % 128 != 0 (one-sided sweep, exact and estimated cap): their rows
    concatenate to the full-range build (symmetric sweep)"""
    V, r, a = case_c_shards()
    N = len(V)
    full_ref = orc.rball_brute(V, r)
    _check_path("c-full", V, r, 0, N, full_ref, expect=SYMMETRIC)
    full = _build(gpu, V, r, 0, N)
    _assert_same(full, full_ref, "full range")
    rows, vals = [], []
    for q0, q1 in ((0, a), (a, a + 1), (a + 1, N)):
        ref = orc.rball_brute(V, r, 0, q0, q1)
        _check_path("c-shard", V, r, q0, q1, ref, expect=SHARDED)
        got = _build(gpu, V, r, q0, q1)
        _assert_same(got, ref, "shard [%d, %d)" % (q0, q1))
        rows.append(got[1])
        vals.append(got[2])
    assert np.array_equal(np.concatenate(rows), full[1])
    assert np.concatenate(vals).tobytes() == full[2].tobytes()


_CHILD = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import mpb200
V = np.load(sys.argv[2])
r = float(sys.argv[3])
mpb200.init(0)
NN = mpb200.MetricNN(V)
D = NN.precompute(r).D
mpb200.load().mpb200_synchronize()       # with MPB200_TRACE set, the launches of the build are listed here
np.save(sys.argv[4], np.concatenate([D.colptr, D.rowval]))
np.save(sys.argv[5], D.nzval)
NN.close()
"""


@pytest.mark.gpu
@pytest.mark.parametrize("switch", ["MPB200_SLAB_BLOCK_SORT", "MPB200_TC_FULL", "MPB200_NO_TC"])
def test_k3_switches_match_oracle(gpu, orc, tmp_path, switch):
    """the switches are read once per process: each build runs in a child process of its own.  Its launch trace shows
    whether the tensor-core sweep (tc_rball.cu) ran."""
    V, r, q0, q1, _ = case_g()
    ref = orc.rball_brute(V, r)
    env = {switch, "MPB200_TRACE"}
    expect = {"MPB200_SLAB_BLOCK_SORT": dict(SYMMETRIC, merges={"block32"}),
              "MPB200_TC_FULL": SHARDED,
              "MPB200_NO_TC": {"tc": False, "sweep": "one-sided", "fill": "slab"}}[switch]
    path = _check_path(switch, V, r, q0, q1, ref, env, expect)
    np.save(tmp_path / "V.npy", V)
    rows, vals = tmp_path / "rows.npy", tmp_path / "vals.npy"
    res = subprocess.run([sys.executable, "-c", _CHILD, ROOT, str(tmp_path / "V.npy"), repr(r), str(rows), str(vals)],
                         env=dict(os.environ, **{k: "1" for k in env}), capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "brute_rball.cu" in res.stderr, res.stderr[-2000:]
    assert ("tc_rball.cu" in res.stderr) == path["tc"], res.stderr[-2000:]
    cr = np.load(rows)
    got = (cr[:len(V) + 1], cr[len(V) + 1:], np.load(vals))
    _assert_same(got, ref, switch)
