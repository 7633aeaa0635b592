"""Deterministic synthetic turntable scans (SURVEY.md section 8d).

The reference ships no sample data (it reads `points/object_%05d/view_%02d/points.pcd` from a user
workspace, mvr/src/file_system_model.cpp:256-314), so benches and tests use this generator: a
"bumpy sphere" of radius ~100 mm centred at (0, 0, 900) mm, scanned from V turntable positions about
the axis through that centre with normal (0, -1, 0) -- the reference's default axis direction
(mvr/src/registrator.cpp:86-87) and millimetre scale (mvr/src/parameter_manager.cpp:14).

Everything derives from a counter-based splitmix64 stream, so any (seed, view, index) is reproducible
on any host without carrying data files around.
"""
import numpy as np

CENTER = np.array([0.0, 0.0, 900.0])
AXIS = np.array([0.0, -1.0, 0.0])
PIVOT = CENTER
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(seed, counter):
    """splitmix64 output for state seed + (counter+1)*golden, vectorised over `counter`."""
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (np.asarray(counter, dtype=np.uint64) + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return z


def uniform(seed, counter):
    """Uniform doubles in (0, 1)."""
    return ((splitmix64(seed, counter) >> np.uint64(11)).astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


def _streams(seed, idx, k):
    return [uniform(seed, idx * np.uint64(8) + np.uint64(s)) for s in range(k)]


def rotation_about_axis(angle, axis=AXIS, pivot=CENTER):
    """4x4 double, column-vector convention: T(pivot) R(axis, angle) T(-pivot)
    (Registrator::getRotationMatrix, mvr/src/registrator.cpp:331-342)."""
    a = np.asarray(axis, dtype=np.float64)
    a = a / np.linalg.norm(a)
    c, s = np.cos(angle), np.sin(angle)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    R = c * np.eye(3) + s * K + (1 - c) * np.outer(a, a)
    M = np.eye(4)
    M[:3, :3] = R
    p = np.asarray(pivot, dtype=np.float64)
    M[:3, 3] = p - R @ p
    return M


def bumpy_radius(u):
    theta = np.arccos(np.clip(u[:, 2], -1.0, 1.0))
    phi = np.arctan2(u[:, 1], u[:, 0])
    return 100.0 * (1.0 + 0.15 * np.sin(3.0 * theta) * np.cos(5.0 * phi) + 0.05 * np.sin(11.0 * phi))


def _directions(seed, idx):
    u1, u2 = _streams(seed, idx, 2)
    z = 2.0 * u1 - 1.0
    r = np.sqrt(np.maximum(0.0, 1.0 - z * z))
    ph = 2.0 * np.pi * u2
    return np.stack([r * np.cos(ph), r * np.sin(ph), z], axis=1)


def _gauss3(seed, idx):
    u = [uniform(seed, idx * np.uint64(8) + np.uint64(s)) for s in (2, 3, 4, 5)]
    r0 = np.sqrt(-2.0 * np.log(u[0]))
    r1 = np.sqrt(-2.0 * np.log(u[2]))
    return np.stack([r0 * np.cos(2 * np.pi * u[1]), r0 * np.sin(2 * np.pi * u[1]), r1 * np.cos(2 * np.pi * u[3])], axis=1)


def _xyzw(p):
    out = np.empty((len(p), 4), dtype=np.float32)
    out[:, :3] = p
    out[:, 3] = 1.0
    return out


def full_object(n, seed=0x5EED0000, noise=0.0):
    """n points on the whole bumpy sphere (object frame), n x 4 float32."""
    idx = np.arange(n, dtype=np.uint64)
    u = _directions(seed, idx)
    p = CENTER + u * bumpy_radius(u)[:, None]
    if noise > 0:
        p = p + noise * _gauss3(seed, idx)
    return _xyzw(p)


def turntable_angle(view, n_views):
    """Pose angle of `view` (generalises PointCloud::initRotation, mvr/src/point_cloud.cpp:400-413:
    ((v<7)?-v:12-v)*pi/6 for 12 views)."""
    half = n_views // 2
    return ((-view) if view <= half else (n_views - view)) * (2.0 * np.pi / n_views)


def view_pose(view, n_views):
    """Ground-truth pose of `view` (sensor frame -> frame of view 0) without generating its points."""
    return np.linalg.inv(rotation_about_axis(view * 2.0 * np.pi / n_views))


def random_placement(seed):
    """A seeded arbitrary rigid move of the object about CENTER (4x4 double): a uniform random rotation (unit quaternion of
    four seeded normals) and a translation up to +-200 mm per axis -- the object put back on the table in another pose."""
    g = _gauss3(seed ^ 0x91ACE, np.arange(2, dtype=np.uint64)).reshape(-1)[:4]
    w, x, y, z = g / np.linalg.norm(g)
    Rq = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                   [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                   [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])
    t = 400.0 * uniform(seed ^ 0x7A55, np.arange(3, dtype=np.uint64)) - 200.0
    M = np.eye(4)
    M[:3, :3] = Rq
    M[:3, 3] = CENTER - Rq @ CENTER + t
    return M


def turntable_view(view, n_views, n, noise=0.2, seed=0x5EED0000, partial=True, angles=None, placement=None):
    """Scan `view` of an n_views turntable sequence: (points n x 4 float32 in the sensor frame,
    ground-truth pose 4x4 double mapping them into the frame of view 0).  angles (optional, indexed by view): the table's
    actual turn for each view instead of the ideal view * 2 pi / n_views (a table that steps unevenly).  placement (optional
    4x4 rigid move): the object is moved by it before the table turns (placed on its side, upside down, ...); the pose still
    maps the view into the frame of view 0 of the same placement."""
    s = seed + view
    theta = view * 2.0 * np.pi / n_views if angles is None else float(angles[view])   # the table has turned the object by +theta
    R = rotation_about_axis(theta)
    if placement is not None:
        R = R @ np.asarray(placement, dtype=np.float64)
    kept = []
    have = 0
    start = 0
    while have < n:
        batch = max(1024, int((n - have) * (1.8 if partial else 1.0)) + 64)
        idx = np.arange(start, start + batch, dtype=np.uint64)
        start += batch
        u = _directions(s, idx)
        p = CENTER + u * bumpy_radius(u)[:, None]
        ur = u @ R[:3, :3].T
        p = p @ R[:3, :3].T + R[:3, 3]
        if partial:
            m = ur[:, 2] < 0.2                    # faces the sensor at the origin (looking down +z)
            p, idx = p[m], idx[m]
        if noise > 0:
            p = p + noise * _gauss3(s, idx)
        kept.append(p)
        have += len(p)
    p = np.concatenate(kept)[:n]
    if placement is not None:
        return _xyzw(p), np.linalg.inv(rotation_about_axis(theta))
    return _xyzw(p), np.linalg.inv(R)


def step_errors(n_views, max_deg, seed=0x5EED0000):
    """Seeded per-view turn errors (radians), uniform in [-max_deg, +max_deg] degrees; view 0 has none (it defines the frame)."""
    e = np.deg2rad(max_deg) * (2.0 * uniform(seed ^ 0x57E9, np.arange(n_views, dtype=np.uint64)) - 1.0)
    e[0] = 0.0
    return e


def uneven_angles(n_views, max_deg, seed=0x5EED0000):
    """Turns of a table that steps unevenly: view * 2 pi / n_views + step_errors(...)[view]."""
    return np.arange(n_views) * (2.0 * np.pi / n_views) + step_errors(n_views, max_deg, seed)


def perturbation(seed=0x5EED0000, angle_deg=2.0, trans_mm=2.0):
    """Fixed small rigid error put on every initial guess: rotation about a seeded axis through the
    object centre plus a seeded translation."""
    u = _directions(seed ^ 0xABCDEF, np.arange(2, dtype=np.uint64))
    E = rotation_about_axis(np.deg2rad(angle_deg), axis=u[0], pivot=CENTER)
    E[:3, 3] += trans_mm * u[1]
    return E


def turntable_sequence(n_views, n, noise=0.2, seed=0x5EED0000, angles=None, placement=None):
    """views (list of n x 4 float32), gt poses (list of 4x4 double, view -> frame of view 0); angles, placement: see
    turntable_view."""
    views, poses = [], []
    for v in range(n_views):
        p, T = turntable_view(v, n_views, n, noise=noise, seed=seed, angles=angles, placement=placement)
        views.append(p)
        poses.append(T)
    return views, poses


def nn_sweep_case(m, n, seed=0x5EED0000, noise=0.5, order="random"):
    """Target: m points on the full object; queries: n points of the same distribution (own seed)
    + noise, in 'random' (generation) order or 'morton' pre-sorted order."""
    tgt = full_object(m, seed=seed)
    q = full_object(n, seed=seed + 0x1000, noise=noise)
    if order == "morton":
        lo = tgt[:, :3].min(axis=0)
        ext = float((tgt[:, :3].max(axis=0) - lo).max())
        c = np.clip(((q[:, :3] - lo) * (1023.0 / ext)).astype(np.int64), 0, 1023)
        key = np.zeros(len(q), dtype=np.int64)
        for b in range(10):
            for a in range(3):
                key |= ((c[:, a] >> b) & 1) << (3 * b + a)
        q = q[np.argsort(key, kind="stable")]
    return tgt, q
