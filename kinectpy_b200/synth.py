"""Synthetic three-sensor Azure Kinect scene (SURVEY.md section 8d).

The reference has no data in-tree (its inputs are recordings processed by an
external extractor, ``extract.py:21-24``), so throughput and parity are measured
on a deterministic synthetic room: a closed box with the floor at ``y = +1.2 m``
(y points down, as ``floor_removal.py:65`` assumes), a "person" made of eight
ellipsoids standing on the floor, one master sensor and two sub sensors on a
2.5 m circle around the person at +-40 degrees yaw.  Everything here is plain
numpy and runs on the host; it is input generation, not part of the hot path.

Randomness is a counter-based hash keyed ``(seed, frame, sensor, pixel)`` so a
frame can be regenerated anywhere without state (seed 1234 is the only seed the
reference itself uses, ``train.py:19``).
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

_U64 = np.uint64
_MASK = (1 << 64) - 1


def mix64(z: np.ndarray) -> np.ndarray:
    """splitmix64 finaliser on uint64 arrays (same constants as the kernels)."""
    with np.errstate(over="ignore"):
        z = (z + _U64(0x9E3779B97F4A7C15)).astype(np.uint64)
        z = (z ^ (z >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> _U64(27))) * _U64(0x94D049BB133111EB)
        return z ^ (z >> _U64(31))


def rng_u64(seed: int, a, b) -> np.ndarray:
    """Counter-based draw: mix64(mix64(mix64(seed) + a) + b)."""
    a = np.asarray(a, dtype=np.uint64)
    b = np.asarray(b, dtype=np.uint64)
    with np.errstate(over="ignore"):
        s = mix64(np.asarray(seed & _MASK, dtype=np.uint64))
        return mix64(mix64(s + a) + b)


def _uniform(seed: int, a, b) -> np.ndarray:
    return (rng_u64(seed, a, b) >> _U64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


@dataclass(frozen=True)
class SensorMode:
    name: str
    width: int
    height: int
    fx: float
    fy: float
    cx: float
    cy: float
    shape: str  # "hexagon" (NFOV) or "circle" (WFOV)

    @property
    def pixels(self) -> int:
        return self.width * self.height


NFOV = SensorMode("NFOV", 640, 576, 504.0, 504.0, (640 - 1) / 2.0, (576 - 1) / 2.0 + 12.0, "hexagon")
WFOV = SensorMode("WFOV", 1024, 1024, 295.6, 295.6, (1024 - 1) / 2.0, (1024 - 1) / 2.0, "circle")
MODES = {"NFOV": NFOV, "WFOV": WFOV}

KAPPA = 0.05
ROOM_LO = np.array([-3.0, -1.6, -1.0])
ROOM_HI = np.array([3.0, 1.2, 5.0])
PERSON_CENTRE = np.array([0.0, 0.0, 2.5])


def xy_table(mode: SensorMode) -> np.ndarray:
    """Calibration table float32[H*W, 2]; NaN outside the sensor's FOV mask.

    Same role as the k4a xy-table behind the ``_depth.dat`` layout the
    reference reads (``utils/io.py:15-20``): ``X = xt * Z``, ``Y = yt * Z``.
    """
    v, u = np.meshgrid(np.arange(mode.height, dtype=np.float64), np.arange(mode.width, dtype=np.float64), indexing="ij")
    un = (u - mode.cx) / mode.fx
    vn = (v - mode.cy) / mode.fy
    r2 = un * un + vn * vn
    xt = un * (1.0 + KAPPA * r2)
    yt = vn * (1.0 + KAPPA * r2)
    # FOV mask in normalised image coordinates
    a = (u - (mode.width - 1) / 2.0) / (mode.width / 2.0)
    b = (v - (mode.height - 1) / 2.0) / (mode.height / 2.0)
    if mode.shape == "hexagon":
        ok = (np.abs(b) <= 1.0) & (np.abs(a) <= 1.0 - np.abs(b) / 2.0)
    else:
        ok = a * a + b * b <= 1.0
    tab = np.stack([xt, yt], axis=-1).astype(np.float32)
    tab[~ok] = np.nan
    return tab.reshape(-1, 2)


def _roty(deg: float) -> np.ndarray:
    c, s = math.cos(math.radians(deg)), math.sin(math.radians(deg))
    return np.array([[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]])


def extrinsics(n_sensors: int = 3) -> np.ndarray:
    """Ground-truth ``T_master<-sensor`` float64[S,4,4]; sensor 0 is the master.

    Same convention as ``transformation_master_sub_<i>.npy``
    (``preprocessing/data.py:158-160``): maps sub coordinates into the master frame.
    """
    # +-40 degrees: enough shared surface (fitness ~0.5 at a 2 cm correspondence gate) for point-to-plane
    # ICP to be well conditioned; at +-120 degrees the views only share floor and ceiling and ICP drifts
    yaws = [0.0, 40.0, -40.0, 80.0, -80.0, 120.0][:n_sensors]
    out = np.zeros((n_sensors, 4, 4))
    for i, yaw in enumerate(yaws):
        R = _roty(yaw)
        pos = PERSON_CENTRE + R @ (np.zeros(3) - PERSON_CENTRE)  # rotate master position about the person
        out[i, :3, :3] = R
        out[i, :3, 3] = pos
        out[i, 3, 3] = 1.0
    return out


def perturbed_extrinsic(T: np.ndarray, angle_deg: float = 1.0, shift_mm=(5.0, -5.0, 5.0), unit_scale: float = 1e-3) -> np.ndarray:
    """ICP start: ground truth perturbed by a rotation about (1,1,1)/sqrt(3) and a small shift."""
    k = np.ones(3) / math.sqrt(3.0)
    K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    th = math.radians(angle_deg)
    R = np.eye(3) + math.sin(th) * K + (1 - math.cos(th)) * (K @ K)
    D = np.eye(4)
    D[:3, :3] = R
    D[:3, 3] = np.asarray(shift_mm, dtype=np.float64) * unit_scale  # mm -> cloud unit
    return D @ T


def _person(frame: int):
    """Eight ellipsoids (centre, radii) in metres; sways with period 100 frames."""
    sway = 0.10 * math.sin(2.0 * math.pi * frame / 100.0)
    x0, z0 = PERSON_CENTRE[0] + sway, PERSON_CENTRE[2]
    fl = ROOM_HI[1]
    return [
        ((x0, fl - 1.62, z0), (0.10, 0.12, 0.10)),         # head
        ((x0, fl - 1.15, z0), (0.20, 0.32, 0.13)),         # torso
        ((x0 - 0.29, fl - 1.15, z0), (0.055, 0.30, 0.055)),  # left arm
        ((x0 + 0.29, fl - 1.15, z0), (0.055, 0.30, 0.055)),  # right arm
        ((x0 - 0.10, fl - 0.62, z0), (0.085, 0.24, 0.085)),  # left thigh
        ((x0 + 0.10, fl - 0.62, z0), (0.085, 0.24, 0.085)),  # right thigh
        ((x0 - 0.10, fl - 0.21, z0), (0.065, 0.21, 0.065)),  # left shin
        ((x0 + 0.10, fl - 0.21, z0), (0.065, 0.21, 0.065)),  # right shin
    ]


def _raycast(T_sensor: np.ndarray, frame: int, tab: np.ndarray):
    """First hit along every pixel's ray: distance t (metres along the unnormalised ray, so t * 1000 is Z in mm),
    whether it is one of the person's ellipsoids, and the table's FOV mask."""
    ok = ~np.isnan(tab[:, 0])
    d_s = np.stack([tab[:, 0].astype(np.float64), tab[:, 1].astype(np.float64), np.ones(tab.shape[0])], axis=-1)
    d_s[~ok] = (0.0, 0.0, 1.0)
    R, o = T_sensor[:3, :3], T_sensor[:3, 3]
    d = d_s @ R.T
    # inside an axis-aligned box the first wall hit is the smallest positive exit distance
    with np.errstate(divide="ignore", invalid="ignore"):
        tx = np.where(d > 0, (ROOM_HI - o) / d, np.where(d < 0, (ROOM_LO - o) / d, np.inf))
    t = tx.min(axis=1)
    person = np.zeros(tab.shape[0], dtype=bool)
    for c, r in _person(frame):
        c = np.asarray(c)
        r = np.asarray(r)
        dn = d / r
        on = (o - c) / r
        qa = (dn * dn).sum(1)
        qb = 2.0 * (dn * on).sum(1)
        qc = float((on * on).sum()) - 1.0
        disc = qb * qb - 4.0 * qa * qc
        hit = disc >= 0
        te = np.where(hit, (-qb - np.sqrt(np.where(hit, disc, 0.0))) / (2.0 * qa), np.inf)
        closer = (te > 0) & (te < t)
        t = np.where(closer, te, t)
        person |= closer
    return t, person & ok, ok


def render_depth(mode: SensorMode, T_sensor: np.ndarray, frame: int, sensor: int, seed: int = 1234,
                 noise: bool = True, table: np.ndarray | None = None) -> np.ndarray:
    """One depth image uint16[H*W] in millimetres (Z along the optical axis; 0 = no return)."""
    tab = xy_table(mode) if table is None else table
    t, _, ok = _raycast(T_sensor, frame, tab)
    z_mm = t * 1000.0
    pix = np.arange(tab.shape[0], dtype=np.uint64)
    key_a = np.uint64(frame) * np.uint64(16) + np.uint64(sensor)
    if noise:
        u1 = _uniform(seed, key_a, pix * np.uint64(4) + np.uint64(0))
        u2 = _uniform(seed, key_a, pix * np.uint64(4) + np.uint64(1))
        u3 = _uniform(seed, key_a, pix * np.uint64(4) + np.uint64(2))
        u4 = _uniform(seed, key_a, pix * np.uint64(4) + np.uint64(3))
        g = np.sqrt(-2.0 * np.log(np.maximum(u1, 1e-300))) * np.cos(2.0 * math.pi * u2)
        z_mm = z_mm + g * (1.5 + 0.001 * z_mm)
        fly = u3 < 0.003
        z_mm = np.where(fly, z_mm * (0.6 + 0.35 * u4), z_mm)
        drop = (u3 >= 0.003) & (u3 < 0.023)
    else:
        drop = np.zeros(tab.shape[0], dtype=bool)
    z = np.rint(z_mm)
    z = np.where(ok & ~drop & (z > 0) & (z < 65535), z, 0.0)
    return z.astype(np.uint16)


FAR_WALL_M = 4.0     # a wall pixel at least this far away can be part of the false-positive patch


def render_segmentation(mode: SensorMode, T_sensor: np.ndarray, frame: int, sensor: int, seed: int = 1234,
                        table: np.ndarray | None = None) -> np.ndarray:
    """The segmentation image that goes with ``render_depth``: uint8[H*W, 3], non-black where a pixel's first hit is
    the person, black elsewhere -- the ``_seg`` image ``DataProcessor`` crops with (preprocessing/data.py:165-178).
    Two seeded defects exercise each rule of the crop: about 3 % of the person pixels have one or two zero channels
    (a pixel is person only when all three channels are non-zero), and a patch of the image that sees a far wall
    (more than FAR_WALL_M away) is marked as person (the median gate has to remove it)."""
    tab = xy_table(mode) if table is None else table
    t, person, ok = _raycast(T_sensor, frame, tab)
    n = tab.shape[0]
    pix = np.arange(n, dtype=np.uint64)
    key_a = np.uint64(frame) * np.uint64(16) + np.uint64(sensor) + np.uint64(1 << 40)
    u = [_uniform(seed, key_a, pix * np.uint64(4) + np.uint64(k)) for k in range(4)]
    rgb = np.zeros((n, 3), dtype=np.uint8)
    shade = (np.stack(u[:3], axis=1) * 200.0 + 40.0).astype(np.uint8)      # 40..239 in every channel
    rgb[person] = shade[person]
    # defect 1: one or two zero channels on a few person pixels
    bad = person & (u[3] < 0.03)
    zero_a = (u[3] * 1000.0).astype(np.int64) % 3
    rows = np.flatnonzero(bad)
    rgb[rows, zero_a[rows]] = 0
    two = rows[(rows % 2) == 0]
    rgb[two, (zero_a[two] + 1) % 3] = 0
    # defect 2: a false-positive patch on a far wall, in a fixed window of the image (an eighth of its width and height,
    # right of and above the centre)
    v, c = np.divmod(np.arange(n), mode.width)
    window = (c >= (5 * mode.width) // 8) & (c < (6 * mode.width) // 8) & (v >= (3 * mode.height) // 8) & (v < (4 * mode.height) // 8)
    patch = ok & ~person & (t > FAR_WALL_M) & window
    rgb[patch] = (200, 180, 160)
    return rgb


def render_sequence(mode: SensorMode, n_frames: int, n_sensors: int = 3, seed: int = 1234, first_frame: int = 0,
                    noise: bool = True):
    """depth uint16[F,S,P], table float32[S,P,2], extrinsics float64[S,4,4] (metres)."""
    tab = xy_table(mode)
    T = extrinsics(n_sensors)
    depth = np.empty((n_frames, n_sensors, mode.pixels), dtype=np.uint16)
    for f in range(n_frames):
        for s in range(n_sensors):
            depth[f, s] = render_depth(mode, T[s], first_frame + f, s, seed, noise, tab)
    tables = np.repeat(tab[None], n_sensors, axis=0).copy()
    return depth, tables, T


def scale_extrinsics(T: np.ndarray, unit_scale: float) -> np.ndarray:
    """Extrinsics in metres -> the unit the cloud is produced in (1e-3 -> metres, 1.0 -> millimetres)."""
    out = np.array(T, dtype=np.float64, copy=True)
    out[..., :3, 3] *= (unit_scale / 1e-3)
    return out
