"""Inputs of the pass-by-pass ICP tests (``test_oracle_icp_passes.py`` on the CPU, ``test_gpu_icp_passes.py`` on the
device): a bumpy textured surface with analytic normals, and constructed clouds for the gate, ties, NaN rows and
degenerate systems.  Every builder is seeded and returns float32 clouds."""
import math

import numpy as np


def rot(ax, ay, az):
    cx, sx, cy, sy, cz, sz = math.cos(ax), math.sin(ax), math.cos(ay), math.sin(ay), math.cos(az), math.sin(az)
    R = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]]) @ np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]]) @ \
        np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    T = np.eye(4)
    T[:3, :3] = R
    return T


def about(Rt, centre, t):
    """The rotation of Rt about `centre`, then the translation t."""
    T = Rt.copy()
    T[:3, 3] = centre - Rt[:3, :3] @ centre + t
    return T


def surface(n, seed):
    """n points of z = 0.08 sin(3x) cos(2y) + 0.05 x y on [-1, 1]², their unit normals and a grey texture."""
    r = np.random.default_rng(seed)
    u = r.uniform(-1, 1, (n, 2))
    x, y = u[:, 0], u[:, 1]
    z = 0.08 * np.sin(3 * x) * np.cos(2 * y) + 0.05 * x * y
    fx = 0.24 * np.cos(3 * x) * np.cos(2 * y) + 0.05 * y
    fy = -0.16 * np.sin(3 * x) * np.sin(2 * y) + 0.05 * x
    nrm = np.stack([-fx, -fy, np.ones(n)], axis=1)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    g = 0.5 + 0.2 * np.sin(9 * x) * np.cos(7 * y) + 0.1 * np.cos(5 * x + 4 * y)
    col = np.stack([g, 0.9 * g, 1.1 * g], axis=1)
    return np.stack([x, y, z], axis=1), nrm, col


def surface_pair(n_src, seed=0, n_tgt=None, unit=1.0, offset=0.0):
    """Target: a surface of about n_src points (at least 64); source: another sample of the same surface (noise of a
    tenth of the spacing) moved off by a small rigid motion.  max_corr is three times the target's spacing, the motion
    half of it, so most points find a partner and the run converges.  ``unit`` scales every length (1000: millimetres),
    ``offset`` shifts both clouds by that many units along (1, 1, 1)."""
    n_tgt = max(n_src, 64) if n_tgt is None else n_tgt
    tp, tn, tc = surface(n_tgt, seed)
    sp, _, sc = surface(n_src, seed + 1000)
    h = 2.0 / math.sqrt(n_tgt)
    r = np.random.default_rng(seed + 7)
    sp = sp + r.normal(0, 0.1 * h, sp.shape)
    D = rot(*(r.uniform(-1, 1, 3) * 0.25 * h))
    D[:3, 3] = r.uniform(-1, 1, 3) * 0.25 * h
    sp = sp @ D[:3, :3].T + D[:3, 3]
    off = np.full(3, offset, np.float64)
    return {"src": ((sp + off / unit) * unit).astype(np.float32), "src_col": sc.astype(np.float32),
            "tgt": ((tp + off / unit) * unit).astype(np.float32), "tgt_n": tn.astype(np.float32),
            "tgt_col": tc.astype(np.float32), "max_corr": 3.0 * h * unit, "unit": unit, "init": np.eye(4)}


# ---------------------------------------------------------------------------------------------------------- the gate
# Lattice 0, 20, 40, 60 on every axis, max_corr = 15, r² = 225 exactly, with integer offsets of length exactly 15:
# (15, 0, 0) beyond a face, (12, 9, 0) beyond an edge, (10, 10, 5) beyond a corner.  Every coordinate is exact in
# float32 and every d² exact in double, so "at the gate" is d² == r² exactly; one float32 ulp of the largest offset
# component inwards (at the source's coordinate) is strictly inside.
GATE = 15.0
ULP15 = 2.0 ** -20           # float32 spacing in [8, 16)
FAR = [(1e3, 1e3, 1e3), (-1e6, 2e6, 1e6), (1e6, -1e6, -3e6)]


def _offsets():
    """Unit direction d in {-1, 0, 1}³ \\ 0 -> an integer offset of length 15 with the signs of d (largest first)."""
    out = []
    for d in np.ndindex(3, 3, 3):
        d = np.array(d) - 1
        nz = np.flatnonzero(d)
        if len(nz) == 0:
            continue
        mag = {1: (15,), 2: (12, 9), 3: (10, 10, 5)}[len(nz)]
        o = np.zeros(3)
        o[nz] = np.array(mag, np.float64) * d[nz]
        out.append((d, o, nz[0]))
    return out


def gate_case(seed=0):
    r = np.random.default_rng(seed)
    g = np.arange(4) * 20.0
    tgt = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    tgt = tgt[r.permutation(len(tgt))]
    src = []
    for d, o, big in _offsets():
        # the lattice point on the face / edge / corner the direction leaves by (inner coordinates: 20 or 40)
        base = np.where(d < 0, 0.0, np.where(d > 0, 60.0, 20.0 + 20.0 * r.integers(0, 2, 3)))
        src.append(base + o)                                    # exactly at the gate: excluded
        inner = (base + o).astype(np.float32)
        inner[big] = np.nextafter(inner[big], np.float32(base[big]))
        src.append(inner.astype(np.float64))                    # one float32 ulp inside: included
        src.append(base + 0.5 * o)                              # well inside
        src.append(base + 1.25 * o)                             # beyond the gate
    src += FAR
    src = np.array(src)
    src = src[r.permutation(len(src))]
    nrm = r.normal(size=tgt.shape)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return {"src": src.astype(np.float32), "tgt": tgt.astype(np.float32), "tgt_n": nrm.astype(np.float32),
            "max_corr": GATE, "unit": 1.0, "init": np.eye(4)}


def one_point_target():
    """A target of one point; one source point exactly at the gate, one an ulp inside, one well inside, two far."""
    src = [(15.0, 0, 0), (0, 12.0 - ULP15, -9.0), (3.0, 4.0, 0.0), (10.0, -10.0, 5.0), (1e3, 0, 0), (0, 0, -1e6)]
    return {"src": np.array(src, np.float32), "tgt": np.zeros((1, 3), np.float32),
            "tgt_n": np.array([[0.6, 0.0, 0.8]], np.float32), "max_corr": GATE, "unit": 1.0, "init": np.eye(4)}


# ---------------------------------------------------------------------------------------------------------- ties
def ties_case(seed=0):
    """Target lattice (spacing 2) whose every point appears twice under unrelated indices, plus sources at the
    cell centres of the lattice (d² = 3 to eight targets, sixteen rows) and near lattice points (two equal rows).
    Per-index random normals: a partner chosen by the wrong tie rule changes J by O(1)."""
    r = np.random.default_rng(seed)
    g = np.arange(6) * 2.0
    lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    tgt = np.concatenate([lat, lat])
    tgt = tgt[r.permutation(len(tgt))]
    c = np.arange(5) * 2.0 + 1.0
    centres = np.stack(np.meshgrid(c, c, c, indexing="ij"), -1).reshape(-1, 3)
    near = lat + r.integers(-4, 5, lat.shape) / 16.0
    src = np.concatenate([centres, near])
    src = src[r.permutation(len(src))]
    nrm = r.normal(size=tgt.shape)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return {"src": src.astype(np.float32), "tgt": tgt.astype(np.float32), "tgt_n": nrm.astype(np.float32),
            "max_corr": 2.0, "unit": 1.0, "init": np.eye(4)}


# ---------------------------------------------------------------------------------------------------------- NaN rows
def nan_case(n=3000, seed=3):
    c = surface_pair(n, seed)
    c["src"][::7] = np.nan
    c["tgt"][5::11] = np.nan
    return c


# ---------------------------------------------------------------------------------------------------------- degenerate
def planar_case():
    """Target on the plane z = 0.5 with the shared normal (0, 0, 1), source on the same plane (dyadic coordinates):
    every residual is exactly 0, so Jᵀr = 0 and the update is the identity."""
    r = np.random.default_rng(5)
    tgt = np.zeros((400, 3))
    tgt[:, :2] = r.integers(-64, 65, (400, 2)) / 64.0
    tgt[:, 2] = 0.5
    src = tgt[:300].copy()
    src[:, :2] += r.integers(-2, 3, (300, 2)) / 256.0
    nrm = np.tile([0.0, 0.0, 1.0], (400, 1))
    return {"src": src.astype(np.float32), "tgt": tgt.astype(np.float32), "tgt_n": nrm.astype(np.float32),
            "max_corr": 0.125, "unit": 1.0, "init": np.eye(4)}


def few_matches_case(nmatch, seed=11):
    """A surface pair cut down so that exactly `nmatch` source points have a partner in pass 0 (the others far)."""
    c = surface_pair(400, seed)
    r = np.random.default_rng(seed)
    keep = r.choice(len(c["src"]), nmatch, replace=False)
    far = np.array(FAR[:2], np.float32)
    c["src"] = np.concatenate([c["src"][keep], far])
    return c


def collinear_case(axis_aligned):
    """Point-to-point on matches along one line (rank-1 cross-covariance): along the x axis the cross-covariance
    has exact zeros, along a general direction it is rank 1 to rounding."""
    r = np.random.default_rng(21)
    d = np.array([1.0, 0.0, 0.0]) if axis_aligned else np.array([0.48, -0.64, 0.6])
    tgt = np.outer(np.arange(-40, 41) / 32.0, d)
    src = np.outer((np.arange(-40, 41)[r.permutation(81)[:30]] + 0.25) / 32.0, d) + (0 if axis_aligned else 0.003)
    return {"src": src.astype(np.float32), "tgt": tgt.astype(np.float32), "max_corr": 0.1, "unit": 1.0, "init": np.eye(4)}


def coplanar_reflection_case():
    """Point-to-point with coplanar matches whose best orthogonal map is a reflection: the source is the target's
    mirror image through the plane's in-plane axis, so the unconstrained SVD solution has det -1."""
    r = np.random.default_rng(23)
    tgt = np.zeros((200, 3))
    tgt[:, :2] = r.uniform(-1, 1, (200, 2))
    tgt[:, 0] *= 0.2
    tgt[:, 0] += 0.05 * np.sign(tgt[:, 1])
    src = tgt.copy()
    src[:, 0] = -src[:, 0] + 0.002
    return {"src": src.astype(np.float32), "tgt": tgt.astype(np.float32), "max_corr": 0.3, "unit": 1.0, "init": np.eye(4)}
