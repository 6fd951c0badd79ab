"""The per-call neighbour search (kp_knn, kp_sor_mask, kp_radius_mask, kp_estimate_normals and the ICP target grid) on
every level and hand-over of kp_grid.cu, held to a float64 brute force.

The search has four paths: the thread-per-query histogram kernel (level 0, 32 or 64 bins), the warp-per-query
best-first kernel on a coarser grid (level 1, profile family ``knn_level1``), the warp-per-query ring expansion with its
linear-scan fallback (``knn_stragglers``), and two ways to find a cell (a cell map, or an open-addressing hash for grids
of more than 2^27 cells).  Each path must return the exact double-precision answer.  Every case here states which path
it is written for and checks, from the profile counts and the ``KP_DEBUG_KNN`` tallies, that it got there: a case
that reaches nothing fails.  Every GPU case runs once on the cell map and once on the hash (``KP_GRID_FORCE_HASH=1``).

Reference: ``d2 = (dx*dx + dy*dy) + dz*dz`` in float64 on the float32 coordinates (numpy does not contract to FMA),
ordered by (d2, index); the hybrid cap is strict, ``d2 < radius * radius`` with the square taken in double; NaN rows
are never returned and a NaN query gets count 0, index -1 and d2 = +inf.  The CPU tests at the end pin this brute
force against the oracle before any GPU run.
"""
import math
import re

import numpy as np
import pytest

import gpu_helpers as G
from conftest import make_surface_cloud

LEVEL0_FAMILY, LEVEL1_FAMILY, STRAG_FAMILY = "knn_level0", "knn_level1", "knn_stragglers"
HASH_CELLS = 134217728          # more cells than this: the grid is a hash (kp_grid_build)
WARP_KMAX = 4032                # largest k whose per-warp buffer (4 warps x next_pow2(k + 64) x 12 bytes) fits 200 KB
KP_E_ARG, KP_E_RANGE = -1, -3


# ------------------------------------------------------------------------------------------------ reference
def brute_knn(pts, k, radius=0.0, rows=None, chunk_elems=1 << 23):
    """Exact kNN (hybrid when radius > 0) of the self-queries `rows` (default: all) against pts, float64."""
    P = np.asarray(pts, np.float32).astype(np.float64)
    n = P.shape[0]
    rows = np.arange(n) if rows is None else np.asarray(rows)
    nq = rows.shape[0]
    idx = np.full((nq, k), -1, np.int32)
    d2 = np.full((nq, k), np.inf)
    cnt = np.zeros(nq, np.int32)
    if n == 0 or nq == 0:
        return idx, d2, cnt
    r2 = radius * radius if radius > 0 else 0.0
    valid = ~np.isnan(P[:, 0])
    kk = min(k, n)
    step = max(1, chunk_elems // n)
    for s in range(0, nq, step):
        r = rows[s:s + step]
        q = P[r]
        dx = q[:, None, 0] - P[None, :, 0]
        dy = q[:, None, 1] - P[None, :, 1]
        dz = q[:, None, 2] - P[None, :, 2]
        d = (dx * dx + dy * dy) + dz * dz
        ok = valid[None, :] & ~np.isnan(q[:, 0])[:, None]
        if r2 > 0:
            ok &= d < r2
        d[~ok] = np.inf
        v = np.partition(d, kk - 1, axis=1)[:, kk - 1]       # k-th smallest: the answer lies at or below it
        ri, ci = np.nonzero((d <= v[:, None]) & ok)
        dv = d[ri, ci]
        o = np.lexsort((ci, dv, ri))                         # by row, then (d2, index)
        ri, ci, dv = ri[o], ci[o], dv[o]
        pos = np.arange(ri.shape[0]) - np.searchsorted(ri, np.arange(r.shape[0]))[ri]
        sel = pos < k
        idx[s + ri[sel], pos[sel]] = ci[sel]
        d2[s + ri[sel], pos[sel]] = dv[sel]
        cnt[s:s + r.shape[0]] = np.bincount(ri[sel], minlength=r.shape[0])
    return idx, d2, cnt


def brute_radius_count(pts, radius, chunk_elems=1 << 23):
    """Points (itself included) with d2 < radius * radius of every self-query; NaN queries count 0."""
    P = np.asarray(pts, np.float32).astype(np.float64)
    n = P.shape[0]
    r2 = radius * radius
    valid = ~np.isnan(P[:, 0])
    out = np.zeros(n, np.int32)
    step = max(1, chunk_elems // max(n, 1))
    for s in range(0, n, step):
        q = P[s:s + step]
        d = ((q[:, None, 0] - P[None, :, 0]) ** 2 + (q[:, None, 1] - P[None, :, 1]) ** 2) + (q[:, None, 2] - P[None, :, 2]) ** 2
        out[s:s + step] = ((d < r2) & valid[None, :]).sum(1)
    out[~valid] = 0
    return out


def reference_normals(pts, idx, cnt):
    """Normals from a neighbour set: cumulants summed in ascending neighbour order, covariance E[xx] - E[x]E[x], the
    eigenvector of the smallest eigenvalue (np.linalg.eigh).  Returns (normals, eigenvalues ascending)."""
    P = np.asarray(pts, np.float32).astype(np.float64)
    n, k = idx.shape
    sm = np.zeros((n, 9))
    for t in range(k):
        on = t < cnt
        j = np.where(on, idx[:, t], 0)
        x, y, z = P[j, 0], P[j, 1], P[j, 2]
        for c, v in enumerate((x, y, z, x * x, x * y, x * z, y * y, y * z, z * z)):
            sm[:, c] += np.where(on, v, 0.0)
    sm /= np.maximum(cnt, 1)[:, None]
    cov = np.empty((n, 3, 3))
    cov[:, 0, 0] = sm[:, 3] - sm[:, 0] * sm[:, 0]
    cov[:, 0, 1] = cov[:, 1, 0] = sm[:, 4] - sm[:, 0] * sm[:, 1]
    cov[:, 0, 2] = cov[:, 2, 0] = sm[:, 5] - sm[:, 0] * sm[:, 2]
    cov[:, 1, 1] = sm[:, 6] - sm[:, 1] * sm[:, 1]
    cov[:, 1, 2] = cov[:, 2, 1] = sm[:, 7] - sm[:, 1] * sm[:, 2]
    cov[:, 2, 2] = sm[:, 8] - sm[:, 2] * sm[:, 2]
    w, V = np.linalg.eigh(cov)
    return V[:, :, 0], w


def separated(w):
    """The smallest eigenvalue is well separated: its gap to the next one is at least 1e-4 of the largest.  The normal is
    then fixed by the covariance to far better than the 1e-6 bar (both sides sum the same cumulants in the same order);
    below that gap the two eigen solvers (analytic on the device, LAPACK here) may pick different vectors of a
    near-degenerate pair.  On these scenes it excludes at most a handful of points with 3 or 4 nearly collinear
    neighbours."""
    return (w[:, 2] > 0) & (w[:, 1] - w[:, 0] > 1e-4 * w[:, 2])


# ------------------------------------------------------------------------------------------------ scenes
def with_nan_rows(pts, every, start=3):
    pts = pts.copy()
    pts[start::every] = np.nan
    return pts


def surface(n, seed):
    """Sheets with 2 % isolated points (uniform in a cube larger than the sheets) and a NaN row every 53."""
    return with_nan_rows(make_surface_cloud(n, seed=seed, outliers=0.02), 53)


def lattice(m=13):
    """Integer coordinates at scale 1: d2 == r2 ties for radius 1, sqrt(2) and 2; a NaN row every 97."""
    g = np.stack(np.meshgrid(np.arange(m), np.arange(m), np.arange(m), indexing="ij"), -1).reshape(-1, 3)
    r = np.random.default_rng(5)
    return with_nan_rows(g[r.permutation(len(g))].astype(np.float32), 97)


def two_clusters(seed=21, n=6000):
    """Two dense clusters 10 m apart with lone points on the line between them: a lone point's cube of k candidates is
    more than 7 coarse cells wide (level 1 hands it on: "cube > 7") and the ring search ends in its linear scan."""
    r = np.random.default_rng(seed)
    a = r.normal(0, 0.05, (n // 2, 3))
    b = r.normal(0, 0.05, (n // 2, 3)) + [10.0, 0, 0]
    lone = np.stack([np.linspace(1.0, 9.0, 9), r.uniform(-0.3, 0.3, 9), r.uniform(-0.3, 0.3, 9)], 1)
    pts = np.concatenate([a, lone, b]).astype(np.float32)
    return pts[r.permutation(len(pts))]


def pile_scene(pile, seed):
    """`pile` identical points in a corner of a surface cloud, away from its sheets."""
    base = make_surface_cloud(6000, seed=seed, outliers=0.01)
    pts = np.concatenate([base, np.tile(np.array([[1.3, -1.3, 1.3]], np.float32), (pile, 1))])
    perm = np.random.default_rng(seed).permutation(len(pts))
    return pts[perm]


def sparse_with_pile(pile=65600, seed=41):
    r = np.random.default_rng(seed)
    base = r.uniform(0, 1, (3000, 3)).astype(np.float32)
    pts = np.concatenate([base, np.full((pile, 3), 0.5, np.float32)])
    return pts[r.permutation(len(pts))]


def far_return(seed=51):
    """A metre-scale cloud plus one return about 1 km away: at a 5 cm cell the grid has ~10^12 cells."""
    pts = make_surface_cloud(8000, seed=seed, outliers=0.01)
    pts[17] = [600.0, 580.0, 590.0]
    return pts


def grid_cells(pts, cell):
    """Cell count of kp_grid_build's layout for this cloud and cell."""
    P = np.asarray(pts, np.float32)
    ok = ~np.isnan(P[:, 0])
    ext = P[ok].max(0).astype(np.float64) - P[ok].min(0).astype(np.float64)
    while np.any(ext / cell > 2000000.0):
        cell *= 2.0
    return float(np.prod(np.floor(ext * (1.0 / cell)) + 2))


_REF = {}


def cached(key, fn):
    if key not in _REF:
        _REF[key] = fn()
    return _REF[key]


# ------------------------------------------------------------------------------------------------ evidence
class Evidence:
    def __init__(self, prof, err):
        self.prof, self.err = prof, err
        self.level0_uncertified = sum(int(m) for m in re.findall(r"level-0 uncertified=(\d+)", err))
        self.level1_uncertified = sum(int(m) for m in re.findall(r"level-1 cell=\S+ uncertified=(\d+)", err))
        self.cells = [float(m) for m in re.findall(r" cell=(\S+) level-0", err)]
        self.handover = dict.fromkeys(("cube", "no-bound", "ball", "bin", "short", "scatter", "order", "uncertified"), 0)
        pat = (r"hand-overs: cube>\d+ (\d+), no-bound (\d+), ball>15 (\d+), bin>cap (\d+), short (\d+), scatter (\d+), "
               r"order (\d+), uncertified (\d+)")
        for m in re.findall(pat, err):
            for key, v in zip(self.handover, m):
                self.handover[key] += int(v)

    def calls(self, family):
        return self.prof.get(family, {}).get("calls", 0)

    def __repr__(self):
        return ("level0=%d level1=%d strag=%d | level-0 uncertified %d, level-1 uncertified %d | hand-overs %s"
                % (self.calls(LEVEL0_FAMILY), self.calls(LEVEL1_FAMILY), self.calls(STRAG_FAMILY),
                   self.level0_uncertified, self.level1_uncertified, self.handover))


@pytest.fixture(params=[False, True], ids=["cellmap", "hash"])
def grid_mode(request, monkeypatch):
    """Every case once on the cell map and once on the open-addressing hash."""
    if request.param:
        monkeypatch.setenv("KP_GRID_FORCE_HASH", "1")
    else:
        monkeypatch.delenv("KP_GRID_FORCE_HASH", raising=False)
    return "hash" if request.param else "cellmap"


@pytest.fixture
def probe(ctx, monkeypatch, capfd):
    """probe(fn) -> (fn(), Evidence): the profile counts and KP_DEBUG_KNN tallies of the calls fn makes.  The shared
    context's profiler is switched off again afterwards."""
    def run(fn):
        monkeypatch.setenv("KP_DEBUG_KNN", "1")
        capfd.readouterr()
        ctx.profile(True)
        try:
            out = fn()
            prof = ctx.profile_read()
        finally:
            ctx.profile(False)
            monkeypatch.delenv("KP_DEBUG_KNN", raising=False)
        ev = Evidence(prof, capfd.readouterr().err)
        print(ev)
        return out, ev
    return run


def assert_knn_equal(got, ref, rows=None):
    gi, gd, gc = got
    if rows is not None:
        gi, gd, gc = gi[rows], gd[rows], gc[rows]
    ri, rd, rc = ref
    assert np.array_equal(gc, rc), "counts differ at rows %s" % np.flatnonzero(gc != rc)[:10]
    assert np.array_equal(gi, ri), "indices differ at rows %s" % np.flatnonzero((gi != ri).any(1))[:10]
    assert np.array_equal(gd, rd)


# ------------------------------------------------------------------------------------------------ hybrid self-queries
# (radius, cell hint): below the typical k-th distance with the default cell (= the radius: the cap binds, and a query
# with fewer than k points inside it leaves level 0 through the all-candidates exit); above it; above it with a cell a
# quarter of the radius (the 27-cell block, not the cap, bounds level 0)
HYBRID = [("below", 0.03, 0.0), ("above", 0.15, 0.0), ("block", 0.15, 0.0375)]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 30, 64])
@pytest.mark.parametrize("name,radius,hint", HYBRID, ids=[h[0] for h in HYBRID])
def test_hybrid_self_queries_exact(ctx, probe, grid_mode, name, radius, hint, k):
    pts = cached("surface", lambda: surface(9000, 61))
    ref = cached(("hyb", name, k), lambda: brute_knn(pts, k, radius))
    got, ev = probe(lambda: G.knn(ctx, pts, k, radius=radius, cell_hint=hint))
    assert_knn_equal(got, ref)
    short = int(((ref[2] < k) & ~np.isnan(pts[:, 0])).sum())
    assert ev.calls(LEVEL0_FAMILY) == 1
    if name == "below":
        # more short queries than level 0 left uncertified: the rest can only have ended at `all && cap_binding`
        assert short > len(pts) // 2 and ev.level0_uncertified < short
    elif name == "block":
        # the cap is not binding: every short query must leave level 0 (the block cannot prove it is complete)
        assert ev.level0_uncertified >= short > 0
        # level 1's cube holds k points but fewer than k inside the cap, and does not cover the cap ball: "no-bound"
        assert ev.calls(LEVEL1_FAMILY) == 1 and ev.handover["no-bound"] > 0 and ev.calls(STRAG_FAMILY) == 1


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 30, 64])
@pytest.mark.parametrize("radius", [1.0, math.sqrt(2.0), 2.0], ids=["r1", "rsqrt2", "r2"])
def test_hybrid_lattice_ties_at_the_cap(ctx, probe, grid_mode, radius, k):
    pts = cached("lattice", lattice)
    ref = cached(("lat", radius, k), lambda: brute_knn(pts, k, radius))
    got, ev = probe(lambda: G.knn(ctx, pts, k, radius=radius))
    assert_knn_equal(got, ref)
    r2 = radius * radius
    # the cap really separates equal distances: lattice neighbours at d2 == 1, 2 or 4 sit on it or just inside it
    on_cap = {1.0: 1.0, math.sqrt(2.0): 2.0, 2.0: 4.0}[radius]
    assert (on_cap < r2) == (radius == math.sqrt(2.0))
    assert (ref[1] == on_cap).any() == (radius == math.sqrt(2.0))
    assert ev.calls(LEVEL0_FAMILY) == 1


def shells(radius, ncent, seed=17):
    """40 points on a sphere around each of `ncent` centres 0.3 apart, rounded to float32: the double d2 of a centre's
    shell spreads over ~1e-6 of radius^2, the resolution at which the fp32 binning of level 0 can misorder it."""
    r = np.random.default_rng(seed)
    g = np.stack(np.meshgrid(np.arange(10), np.arange(10), np.arange(6), indexing="ij"), -1).reshape(-1, 3)
    centres = g[:ncent] * 0.3 + 0.05
    u = r.normal(size=(ncent, 40, 3))
    u /= np.linalg.norm(u, axis=2, keepdims=True)
    pts = np.concatenate([centres, (centres[:, None, :] + radius * u).reshape(-1, 3)]).astype(np.float32)
    perm = r.permutation(len(pts))
    return pts[perm], np.flatnonzero(perm < ncent)          # the cloud and the rows of the centres


CAP = 0.1
# with the default cell the cap binds level 0: 32 bins over r2 * (1 + 2e-6); the lower edge of bin 16 in d2
EDGE16 = math.sqrt(15.5 / float(np.float32(31.0 / (CAP * CAP * (1.0 + 2e-6)))))
SHELLS = [("cap", CAP, 120, 8), ("cap", CAP, 120, 30), ("cap", CAP, 120, 64),
          ("edge", EDGE16, 600, 18), ("edge", EDGE16, 600, 20), ("edge", EDGE16, 600, 22)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,shell,ncent,k", SHELLS, ids=["%s-k%d" % (s[0], s[3]) for s in SHELLS])
def test_hybrid_within_fp32_rounding(ctx, oracle, probe, grid_mode, name, shell, ncent, k):
    """Shells on the cap: eligible (d2 < r2) and ineligible candidates interleave in fp32 order, and level 0 must notice
    an eligible entry behind an ineligible one (the `closed` rule).  Shells on the lower edge of bin 16: the k-th
    distance sits on a bin edge, with uncollected candidates just above it, and only the certificate's margin keeps a
    candidate binned one bin too high out of the answer."""
    pts, centres = cached(("shells", name), lambda: shells(shell, ncent))
    rows = np.union1d(centres, np.random.default_rng(k).choice(len(pts), 300, replace=False))
    ref = cached(("shells", name, k), lambda: brute_knn(pts, k, CAP, rows=rows))
    got, ev = probe(lambda: G.knn(ctx, pts, k, radius=CAP))
    assert_knn_equal(got, ref, rows=rows)
    assert_knn_equal(got, cached(("shells", name, k, "oracle"), lambda: oracle.knn(pts, k, radius=CAP)))
    assert ev.level0_uncertified > 0


def f32_d2(q, P):
    """The fp32 squared distance of the histogram kernels (hq_d32: fma(dz, dz, fma(dy, dy, dx * dx)))."""
    d = [(np.float32(q[c]) - P[:, c]).astype(np.float32) for c in range(3)]
    t = (d[0] * d[0]).astype(np.float32)
    t = (d[1].astype(np.float64) * d[1] + t).astype(np.float32)
    return (d[2].astype(np.float64) * d[2] + t).astype(np.float32)


def misordered_pairs(kind, npairs=64, seed=23):
    """Per centre exactly two more points, chosen so that fp32 and double order disagree.  "cap": A with d2 < r2 and B
    with d2 >= r2 but fp32 d2(A) > fp32 d2(B) (B is evaluated first and closes the list before the eligible A).  "edge":
    X in bin 15 and Y in bin 16 of level 0 with d2(Y) < d2(X): at k = 2 the collected k-th entry X lies within rounding
    of the bin edge and only the certificate's margin sends the query on."""
    r = np.random.default_rng(seed)
    scale = np.float32(31.0 / (CAP * CAP * (1.0 + 2e-6)))
    target = CAP * CAP if kind == "cap" else 15.5 / float(scale)
    g = np.stack(np.meshgrid(np.arange(10), np.arange(10), np.arange(6), indexing="ij"), -1).reshape(-1, 3)
    out = []
    for c in (g[:npairs] * 0.3 + 0.05).astype(np.float32):
        u = r.normal(size=(4000, 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        P = (c + np.sqrt(target) * u).astype(np.float32)
        dd = c.astype(np.float64) - P
        d = (dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1]) + dd[:, 2] * dd[:, 2]
        f = f32_d2(c, P)
        if kind == "cap":
            lo, hi = d < CAP * CAP, d >= CAP * CAP
            a, b = np.flatnonzero(lo)[np.argmax(f[lo])], np.flatnonzero(hi)[np.argmin(f[hi])]
            ok = f[a] > f[b]
        else:
            bins = (f.astype(np.float64) * scale + 8388608.0).astype(np.float32).astype(np.float64) - 8388608.0
            lo, hi = bins == 15, bins == 16
            a, b = np.flatnonzero(lo)[np.argmax(d[lo])], np.flatnonzero(hi)[np.argmin(d[hi])]
            ok = d[b] < d[a]
        if ok:
            out.append(np.stack([c, P[a], P[b]]))
    return np.concatenate(out)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,k", [("cap", 8), ("edge", 2)])
def test_hybrid_fp32_misordered_pairs(ctx, probe, grid_mode, kind, k):
    pts = cached(("pairs", kind), lambda: misordered_pairs(kind))
    assert len(pts) >= 3 * 48
    got, ev = probe(lambda: G.knn(ctx, pts, k, radius=CAP))
    assert_knn_equal(got, brute_knn(pts, k, CAP))
    assert ev.level0_uncertified >= 16


# ------------------------------------------------------------------------------------------------ cell hints
@pytest.mark.gpu
def test_cell_hint_never_changes_the_result(ctx, oracle, probe, grid_mode):
    """Hints of 0.1x, 1x and 10x the automatic cell on self-queries: plain kNN, hybrid kNN and SOR.  0.1x starves the
    block (level 1 and the ring search take most queries), 10x floods the level-0 buffer."""
    pts = cached("surface", lambda: surface(9000, 61))
    ref20 = cached(("plain", 20), lambda: brute_knn(pts, 20))
    ref_h = cached(("hyb", "above", 30), lambda: brute_knn(pts, 30, 0.15))
    ref_sor = cached(("sor", 20), lambda: oracle.sor(pts, 20, 2.0))
    _, ev = probe(lambda: G.knn(ctx, pts, 20))
    auto = ev.cells[0]
    seen = {}
    for mult in (0.1, 1.0, 10.0):
        hint = auto * mult
        got, ev = probe(lambda: G.knn(ctx, pts, 20, cell_hint=hint))
        assert_knn_equal(got, ref20)
        seen[mult] = ev
        got, evh = probe(lambda: G.knn(ctx, pts, 30, radius=0.15, cell_hint=hint))
        assert_knn_equal(got, ref_h)
        keep, mean, stats, kept = G.sor(ctx, pts, 20, 2.0, cell_hint=hint)
        assert np.array_equal(mean, ref_sor[1]) and np.array_equal(stats, ref_sor[2]) and np.array_equal(keep, ref_sor[0])
        assert kept == ref_sor[0].sum()
    assert seen[0.1].level0_uncertified > len(pts) // 2 and seen[0.1].calls(STRAG_FAMILY) == 1
    assert seen[10.0].level0_uncertified > len(pts) // 10 and seen[10.0].calls(LEVEL1_FAMILY) == 1


# ------------------------------------------------------------------------------------------------ level-1 hand-overs
@pytest.mark.gpu
def test_level1_cube_overflow_hands_over_to_the_ring_search(ctx, probe, grid_mode):
    pts = cached("clusters", two_clusters)
    for k in (20, 50):
        ref = cached(("clusters", k), lambda: brute_knn(pts, k))
        got, ev = probe(lambda: G.knn(ctx, pts, k))
        assert_knn_equal(got, ref)
        # the lone points 3 m or more from both clusters at least
        assert ev.handover["cube"] >= 5 and ev.calls(LEVEL1_FAMILY) == 1 and ev.calls(STRAG_FAMILY) == 1
        assert ev.level1_uncertified >= 5


@pytest.mark.gpu
def test_level1_bin_overflow_hands_over_to_the_ring_search(ctx, probe, grid_mode):
    """An isolated pile of 200 identical points at k = 20: all 200 share one bin at both levels."""
    pts = cached("pile200", lambda: pile_scene(200, 31))
    ref = cached(("pile200", 20), lambda: brute_knn(pts, 20))
    got, ev = probe(lambda: G.knn(ctx, pts, 20))
    assert_knn_equal(got, ref)
    assert ev.handover["bin"] >= 200 and ev.calls(STRAG_FAMILY) == 1
    pile = np.flatnonzero((pts == np.float32([1.3, -1.3, 1.3])).all(1))
    assert len(pile) == 200 and np.array_equal(got[0][pile], np.tile(np.sort(pile)[:20], (200, 1)))


# ------------------------------------------------------------------------------------------------ 16-bit bin wrap
@pytest.mark.gpu
@pytest.mark.parametrize("k", [20, 60])
def test_pile_of_65600_wraps_a_level0_bin(ctx, oracle, probe, grid_mode, k):
    """65 600 identical points wrap a 16-bit level-0 bin count (to 64).  At k = 20 the wrapped count still exceeds the
    buffer; at k = 60 it fits it, and only the collection count (65 600 puts != 64) can catch the wrap."""
    pts = cached("pile65600", sparse_with_pile)
    pile = np.flatnonzero((pts == 0.5).all(1))
    rest = np.flatnonzero(~(pts == 0.5).all(1))
    got, ev = probe(lambda: G.knn(ctx, pts, k))
    gi, gd, gc = got
    # a pile point: the k lowest pile indices at d2 = 0
    assert np.array_equal(gi[pile], np.tile(pile[:k], (len(pile), 1))) and not gd[pile].any() and (gc[pile] == k).all()
    sample = np.random.default_rng(k).choice(len(pts), 256, replace=False)
    assert_knn_equal(got, cached(("pile65600", k, "brute"), lambda: brute_knn(pts, k, rows=sample)), rows=sample)
    ri, rd, rc = cached(("pile65600", k, "oracle"), lambda: oracle.knn(pts, k, queries=pts[rest]))
    assert_knn_equal(got, (ri, rd, rc), rows=rest)
    assert ev.level0_uncertified >= len(pile) and ev.handover["bin"] >= len(pile)
    if k == 20:
        keep, mean, stats, kept = G.sor(ctx, pts, 20, 1.0)
        rk, rm, rs = cached("pile65600 sor", lambda: oracle.sor(pts, 20, 1.0))
        assert np.array_equal(mean, rm) and np.array_equal(stats, rs) and np.array_equal(keep, rk) and kept == rk.sum()


# ------------------------------------------------------------------------------------------------ k at the limits
@pytest.mark.gpu
def test_largest_k_of_the_warp_buffer(ctx, grid_mode):
    from kinectpy_b200 import KinectPyB200Error
    pts = cached("k4032", lambda: with_nan_rows(make_surface_cloud(5000, seed=71, outliers=0.02), 211))
    ref = cached(("k4032", WARP_KMAX), lambda: brute_knn(pts, WARP_KMAX))
    assert_knn_equal(G.knn(ctx, pts, WARP_KMAX), ref)
    with pytest.raises(KinectPyB200Error) as e:
        G.knn(ctx, pts, WARP_KMAX + 1)
    assert e.value.code == KP_E_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("radius", [0.0, 0.1])
def test_degenerate_clouds(ctx, grid_mode, radius):
    base = make_surface_cloud(40, seed=81)
    cases = [(np.zeros((0, 3), np.float32), 5), (base[:1], 1), (base[:1], 4), (base, 40), (base, 64), (base, 65),
             (base, 100), (np.full((30, 3), np.nan, np.float32), 8), (with_nan_rows(base, 2, 0), 40)]
    for pts, k in cases:
        assert_knn_equal(G.knn(ctx, pts, k, radius=radius), brute_knn(pts, k, radius))


# ------------------------------------------------------------------------------------------------ the hash grid
@pytest.mark.gpu
def test_far_return_reaches_the_hash_without_the_switch(ctx, probe, monkeypatch):
    monkeypatch.delenv("KP_GRID_FORCE_HASH", raising=False)
    pts = far_return()
    assert grid_cells(pts, 0.05 * (1 + 4e-6)) > HASH_CELLS and grid_cells(pts, 0.05 * (1 + 1e-6)) > HASH_CELLS
    got, ev = probe(lambda: G.knn(ctx, pts, 20, radius=0.05))
    assert_knn_equal(got, brute_knn(pts, 20, 0.05))
    assert ev.cells[0] == pytest.approx(0.05 * (1 + 4e-6), rel=1e-5)
    got, ev = probe(lambda: G.knn(ctx, pts, 20, cell_hint=0.05))
    assert_knn_equal(got, brute_knn(pts, 20))
    assert ev.calls(STRAG_FAMILY) == 1            # the far point: ring search, then its linear scan
    _, cnt, _ = G.radius_outlier(ctx, pts, 3, 0.05)
    assert np.array_equal(cnt, brute_radius_count(pts, 0.05))


@pytest.mark.gpu
def test_radius_counts_exact(ctx, grid_mode):
    pts = cached("surface", lambda: surface(9000, 61))
    for nb, r in ((4, 0.03), (20, 0.1)):
        keep, cnt, kept = G.radius_outlier(ctx, pts, nb, r)
        ref = cached(("rcount", r), lambda: brute_radius_count(pts, r))
        assert np.array_equal(cnt, ref) and np.array_equal(keep, (ref > nb).astype(np.uint8)) and kept == (ref > nb).sum()
    lat = cached("lattice", lattice)
    for r in (1.0, math.sqrt(2.0), 2.0):
        _, cnt, _ = G.radius_outlier(ctx, lat, 1, r)
        assert np.array_equal(cnt, brute_radius_count(lat, r))


# ------------------------------------------------------------------------------------------------ normals
@pytest.mark.gpu
@pytest.mark.parametrize("radius,nn", [(0.03, 30), (0.15, 30), (0.15, 64), (0.06, 12)])
def test_normals_on_hybrid_scenes(ctx, grid_mode, radius, nn):
    pts = cached("surface", lambda: surface(9000, 61))
    ri, rd, rc = cached(("hyb-n", radius, nn), lambda: brute_knn(pts, nn, radius))
    ref, w = reference_normals(pts, ri, rc)
    got = G.normals(ctx, pts, radius, nn).astype(np.float64)
    few = rc < 3
    assert few.any() and np.array_equal(got[few], np.tile([0.0, 0.0, 1.0], (few.sum(), 1)))
    sep = separated(w) & ~few
    excluded = int((~sep & ~few).sum())
    print("normals r=%g nn=%d: %d of %d points with >= 3 neighbours excluded (eigenvalue gap)" % (radius, nn, excluded, (~few).sum()))
    assert excluded < 0.01 * (~few).sum()
    dots = np.abs((got[sep] * ref[sep]).sum(1))
    assert (dots > 1 - 1e-6).all(), np.flatnonzero(sep)[dots <= 1 - 1e-6][:10]


# ------------------------------------------------------------------------------------------------ ICP on the hash grid
def icp_scene(oracle, seed):
    tgt = make_surface_cloud(12000, seed=seed, outliers=0.0)
    nrm = oracle.estimate_normals(tgt, 0.08, 30)
    col = np.clip(0.5 + 0.4 * np.sin(7 * tgt[:, :1] + np.array([[0.0, 1.0, 2.0]], np.float32)), 0, 1).astype(np.float32)
    from kinectpy_b200 import synth
    D = synth.perturbed_extrinsic(np.eye(4), angle_deg=0.6, shift_mm=(5, -4, 3), unit_scale=1e-3)
    sel = np.arange(0, len(tgt), 2)
    src = oracle.transform(tgt[sel], np.linalg.inv(D))
    return src, col[sel], tgt, col, nrm


@pytest.mark.gpu
def test_icp_variants_on_the_hash_grid(ctx, oracle, monkeypatch):
    src, scol, tgt, tcol, nrm = cached("icp", lambda: icp_scene(oracle, 91))
    runs = {
        "plane": (lambda: G.icp(ctx, src, tgt, nrm, 0.05, max_iter=30),
                  lambda: oracle.icp_point_to_plane(src, tgt, nrm, 0.05, init=np.eye(4), max_iter=30)),
        "point": (lambda: G.icp_p2p(ctx, src, tgt, 0.05, max_iter=30),
                  lambda: oracle.icp_point_to_point(src, tgt, 0.05, init=np.eye(4), max_iter=30)),
        "colored": (lambda: G.icp_colored(ctx, src, scol, tgt, tcol, nrm, 0.03, max_iter=30),
                    lambda: oracle.icp_colored(src, scol, tgt, tcol, nrm, 0.03, init=np.eye(4), max_iter=30)),
    }
    for name, (gpu, ref) in runs.items():
        monkeypatch.delenv("KP_GRID_FORCE_HASH", raising=False)
        a = gpu()
        monkeypatch.setenv("KP_GRID_FORCE_HASH", "1")
        b = gpu()
        monkeypatch.delenv("KP_GRID_FORCE_HASH", raising=False)
        r = ref()
        assert a["iters"] == b["iters"] and a["ncorr"] == b["ncorr"], name
        assert np.abs(a["T"] - b["T"]).max() < 1e-9, name
        assert b["iters"] == r["iters"] and b["ncorr"] == r["ncorr"], name
        assert np.abs(b["T"] - r["T"]).max() < 1e-4, name


# ------------------------------------------------------------------------------------------------ hash capacity
@pytest.mark.gpu
def test_hash_capacity_beyond_2_31_slots_is_refused(ctx):
    """More than 2^30 points over more than 2^30 cells would need a 2^32-slot hash: the call is refused with
    KP_E_RANGE before any workspace is taken (the 32-bit capacity used to wrap to 0 and loop forever)."""
    torch = pytest.importorskip("torch")
    n = (1 << 30) + 4096
    free, _ = torch.cuda.mem_get_info()
    if free < n * 12 + (4 << 30):
        pytest.skip("needs %.1f GB of free device memory" % ((n * 12 + (4 << 30)) / 1e9))
    from kinectpy_b200 import KinectPyB200Error
    import ctypes as C
    pts = torch.zeros((n, 3), dtype=torch.float32, device="cuda")
    pts[::1024, 0] = torch.arange(0, n, 1024, device="cuda", dtype=torch.float32) * (1100.0 / n)
    pts[1, :] = 1100.0
    torch.cuda.synchronize()
    q = ctx.to_device(np.zeros((1, 3), np.float32))
    idx, d2, cnt = ctx.empty((1, 1), np.int32), ctx.empty((1, 1), np.float64), ctx.empty((1,), np.int32)
    try:
        assert grid_cells(np.array([[0, 0, 0], [1100, 1100, 1100]], np.float32), 1.0) > 2 ** 30
        with pytest.raises(KinectPyB200Error) as e:
            ctx.check(ctx.lib.kp_knn(ctx.handle, C.c_void_p(pts.data_ptr()), n, q.ptr, 1, 1, 0.0, 1.0, idx.ptr, d2.ptr, cnt.ptr))
        assert e.value.code == KP_E_RANGE and "2^31" in str(e.value)
    finally:
        del pts
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ CPU: the reference
def test_brute_force_matches_the_oracle(oracle):
    """The brute force is pinned to the oracle before any GPU run: plain and hybrid, NaN rows, k above the valid count,
    lattice ties at d2 == r2 (radius = sqrt(2) squares to 2.0000000000000004 and admits d2 = 2)."""
    assert math.sqrt(2.0) * math.sqrt(2.0) == 2.0000000000000004
    clouds = [surface(1500, 3), lattice(7), make_surface_cloud(30, seed=4)]
    for pts in clouds:
        for k, radius in ((1, 0.0), (8, 0.0), (33, 0.0), (50, 0.08), (8, 1.0), (30, math.sqrt(2.0)), (64, 2.0)):
            ref = oracle.knn(pts, k, radius=radius)
            assert_knn_equal(brute_knn(pts, k, radius, chunk_elems=1 << 16), ref)
    lat = lattice(7)
    i, d, c = brute_knn(lat, 30, math.sqrt(2.0))
    assert (d == 2.0).any() and c.max() == 19                # self + 6 at d2 = 1 + 12 at d2 = 2
    i, d, c = brute_knn(lat, 30, 2.0)
    assert not (d == 4.0).any() and c.max() == 27            # d2 = 4 is on the cap: excluded
    nan_q = np.isnan(lat[:, 0])
    assert (c[nan_q] == 0).all() and (i[nan_q] == -1).all() and np.isinf(d[nan_q]).all()
    assert not np.isin(np.flatnonzero(nan_q), i).any()       # NaN rows are never returned
    rows = np.array([5, 0, 77])
    full = brute_knn(clouds[0], 12, 0.1)
    part = brute_knn(clouds[0], 12, 0.1, rows=rows)
    assert all(np.array_equal(f[rows], p) for f, p in zip(full, part))
    assert [a.shape for a in brute_knn(np.zeros((0, 3), np.float32), 4)] == [(0, 4), (0, 4), (0,)]
    for kind, k in (("cap", 8), ("edge", 2)):
        pts = misordered_pairs(kind, npairs=16)
        assert_knn_equal(brute_knn(pts, k, CAP), oracle.knn(pts, k, radius=CAP))


def test_brute_radius_count_and_normals_match_the_oracle(oracle):
    for pts in (surface(1500, 6), lattice(7)):
        for r in (0.05, 1.0, math.sqrt(2.0), 2.0):
            _, rc = oracle.radius_outlier(pts, 1, r)
            assert np.array_equal(brute_radius_count(pts, r, chunk_elems=1 << 16), rc)
    pts = surface(3000, 7)
    for radius, nn in ((0.15, 30), (0.06, 12)):
        ri, rd, rc = brute_knn(pts, nn, radius)
        ref, w = reference_normals(pts, ri, rc)
        orc = oracle.estimate_normals(pts, radius, nn).astype(np.float64)
        few = rc < 3
        assert np.array_equal(orc[few], np.tile([0.0, 0.0, 1.0], (few.sum(), 1)))
        sep = separated(w) & ~few
        assert (~sep & ~few).sum() < 0.01 * (~few).sum()
        assert (np.abs((orc[sep] * ref[sep]).sum(1)) > 1 - 1e-6).all()
