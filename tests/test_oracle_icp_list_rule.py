"""The rule by which a batched ICP pass takes a point's partner from the target's neighbour lists (DESIGN §3), held to
brute force in NumPy.  It pins the rule, not the kernel.

A target point t has the list of its normals search (hybrid: d2 < r^2, at most max_nn entries, itself included, canonical
(d2, index) order), cut to L = 12 entries besides t, each with its d2 rounded down to float32, and rho2(t) rounded down
to float32: the d2 of the first entry the cut drops; else r^2 when fewer than max_nn qualified; else the d2 of the
max_nn-th entry.  A source point q whose previous partner is t, at d2(q, t) = delta2 < gate^2, takes the list path when
4 * delta2 * (1 + 1e-6) < rho2(t); it then scans t's list up to the first entry whose stored d2 exceeds that bound.
Whenever it does, its exact partner (brute force over the whole target) must be t or one of the scanned entries, and the
canonical minimum over those candidates must be that partner."""
import numpy as np
import pytest

L = 12


def d2(a, b):
    """Squared distances in double of float32-stored points, summed as kp_d2 does: (dx^2 + dy^2) + dz^2."""
    a = a.astype(np.float64)[:, None, :]
    b = b.astype(np.float64)[None, :, :]
    e = a - b
    return (e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1]) + e[..., 2] * e[..., 2]


def f32_down(x):
    """float32 rounding toward -inf of non-negative doubles."""
    f = np.asarray(x, np.float64).astype(np.float32)
    up = f.astype(np.float64) > x
    f[up] = np.nextafter(f[up], np.float32(-np.inf))
    return f


def lists(tgt, radius, max_nn):
    """Per target point: (list positions, stored d2, rho2) and which of the three rho cases applied."""
    D = d2(tgt, tgt)
    n = len(tgt)
    out, cases = [], {"cut": 0, "cap": 0, "max_nn": 0}
    for p in range(n):
        ok = np.flatnonzero(D[p] < radius * radius)
        order = ok[np.lexsort((ok, D[p, ok]))][:max_nn]            # canonical (d2, index), cut to max_nn
        others = order[order != p]
        if len(others) > L:
            rho, case = D[p, others[L]], "cut"
        elif len(order) < max_nn:
            rho, case = radius * radius, "cap"
        else:
            rho, case = D[p, order[-1]], "max_nn"
        cases[case] += 1
        ent = others[:L]
        out.append((ent, f32_down(D[p, ent]), f32_down(rho)))
    return out, cases


def check_rule(tgt, src, prev, gate, lst):
    """Returns how many points the list decided; asserts the partner every time it does."""
    D = d2(src, tgt)
    n = len(tgt)
    decided = 0
    for i, t in enumerate(prev):
        delta2 = D[i, t]
        ent, ed2, rho = lst[t]
        bound = 4.0 * delta2 * (1.0 + 1e-6)
        if not (delta2 < gate * gate and bound < rho):
            continue
        decided += 1
        ok = np.flatnonzero(D[i] < gate * gate)
        exact = ok[np.lexsort((ok, D[i, ok]))][0]                    # brute force: canonical nearest inside the gate
        scanned = ent[:int(np.searchsorted(ed2, bound, side="right"))]
        cand = np.concatenate(([t], scanned))
        got = cand[np.lexsort((cand, D[i, cand]))][0]
        assert exact == t or exact in scanned, (i, t, exact)
        assert got == exact
        assert exact < n
    return decided


def surface(n, seed):
    """A wavy sheet with 1 mm noise, about 5 mm spacing (float32 storage)."""
    r = np.random.default_rng(seed)
    xy = r.uniform(0.0, 0.25, (n, 2))
    z = 0.02 * np.sin(xy[:, 0] * 40.0) * np.cos(xy[:, 1] * 30.0) + r.normal(0.0, 1e-3, n)
    return np.column_stack([xy, z]).astype(np.float32)


def moved(tgt, m, seed, scale):
    """Source points near the target and the index of a target point near each (the 'previous partner')."""
    r = np.random.default_rng(seed)
    base = r.integers(0, len(tgt), m)
    src = (tgt[base].astype(np.float64) + r.normal(0.0, scale, (m, 3))).astype(np.float32)
    D = d2(src, tgt)
    # the previous partner: the nearest, the second nearest or a random one of the 5 nearest (a pass moves the point)
    near = np.argsort(D, axis=1)[:, :5]
    pick = r.integers(0, 5, m) * (r.random(m) < 0.3)
    return src, near[np.arange(m), pick]


@pytest.mark.parametrize("max_nn", [30, 13, 2, 1])
def test_surface_clouds(max_nn):
    tgt = surface(2500, 1)
    lst, cases = lists(tgt, 0.02, max_nn)
    src, prev = moved(tgt, 2000, 2, 2e-3)
    decided = check_rule(tgt, src, prev, 0.02, lst)
    if max_nn == 30:
        assert cases["cut"] > 0 and cases["cap"] > 0
    if max_nn in (13, 2):
        assert cases["max_nn"] > 0 and cases["cut"] == 0
    if max_nn == 1:
        # the list holds nothing and rho2 is the point's own d2 = 0: nothing is decided
        assert decided == 0
    else:
        assert decided > 0.1 * len(src), decided


def test_sparse_cloud_rho_is_the_radius():
    """Fewer than max_nn points inside the radius everywhere: rho2 = r^2, the whole radius is covered."""
    tgt = surface(300, 3)
    lst, cases = lists(tgt, 0.02, 30)
    assert cases["cap"] > 0.5 * len(tgt)
    src, prev = moved(tgt, 1500, 4, 4e-3)
    assert check_rule(tgt, src, prev, 0.02, lst) > 0


@pytest.mark.parametrize("max_nn", [30, 13, 2])
def test_lattice_with_exact_ties(max_nn):
    """A lattice of about 1 cm (2^-7 m, so that the midpoints are exact in float32): every source point sits at the
    midpoint of two target points (or at the centre of four or eight), so the partner is decided by the index alone, and
    the previous partner is the one with the larger index."""
    h = 2.0 ** -7
    g = np.arange(8, dtype=np.float64) * h
    tgt = np.array(np.meshgrid(g, g, g[:3], indexing="ij")).reshape(3, -1).T.astype(np.float32)
    lst, cases = lists(tgt, 0.02, max_nn)
    half = np.array([[1, 0, 0], [0, 1, 0], [1, 1, 0], [1, 1, 1], [0, 0, 1]]) * (h / 2)
    base = tgt[(tgt[:, 0] < 6.5 * h) & (tgt[:, 1] < 6.5 * h) & (tgt[:, 2] < 1.5 * h)].astype(np.float64)
    src = (base[:, None, :] + half[None]).reshape(-1, 3).astype(np.float32)
    D = d2(src, tgt)
    m = D.min(1, keepdims=True)
    tied = D == m
    assert (tied.sum(1) >= 2).all()
    prev = np.array([np.flatnonzero(row)[-1] for row in tied])         # the tied point with the largest index
    decided = check_rule(tgt, src, prev, 0.02, lst)
    print("lattice, max_nn %d: rho cases %s, %d of %d decided by the list" % (max_nn, cases, decided, len(src)))
    if max_nn == 2:
        # rho = the lattice step = 2 delta exactly: a tied point may sit on that sphere, and the strict test declines
        assert decided == 0
    else:
        assert decided > 0
