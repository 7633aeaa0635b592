"""The two neighbourhood kernels under most of the library, against exact CPU references.

k_normals (csrc/normals.cu) feeds point-to-plane and symmetric ICP, the ring registration's normals batch and the FPFH
keypoints.  Its neighbour lists must equal, bit for bit, a brute-force kNN in the kernel's pinned float32 distance with ties
to the lower index, at k on both sides of the k_normals<16> / k_normals<32> instantiations, on clouds that force the shell
walk past the 3 x 3 x 3 block, the 4096-cell axis cap, the grown-cell grid cap, a single cell, short lists, stacks of
identical points and non-finite points.  Its normals and curvatures are checked against a float64 two-pass covariance and
numpy's eigh (an eigen-solver independent of the kernel's Jacobi), within a tolerance set by each neighbourhood's eigen-gap,
and exactly on planar, collinear and all-identical neighbourhoods.

k_dn_edges / dn_union / dn_find (csrc/denoise.cu) label the radius graph with a lock-free union-find whose roots must be the
components' smallest indices, since the output order depends on it.  The kept indices, in output order, and the noise count
are checked against the components of the radius graph under the kernel's own float64 edge predicate: edges at exactly
triangle_length and one float ulp beyond it, 200k-point chains, one 2M-point component, components of segment_threshold - 1,
segment_threshold and segment_threshold + 1 points, 5000 copies of one point, non-finite points, and grids whose cells were
grown or whose axis was capped to fit the table.
"""
import numpy as np
import pytest

KS = [3, 4, 7, 15, 16, 17, 31, 32]        # both sides of k_normals<16> / k_normals<32> and their edges
MAX_CELLS = 16 * 1024 * 1024              # make_pair_grid's table limit (csrc/api.cu)


# ---- CPU references ---------------------------------------------------------------------------------------------------
def _finite(pts):
    return np.isfinite(pts[:, :3]).all(axis=1)


def knn_reference(pts, k):
    """Brute-force kNN: per point the k finite points of smallest (d2, original index), self included, with d2 the kernel's
    pinned float32 ((dx*dx + dy*dy) + dz*dz) (numpy rounds every operation; it never contracts to FMA).  Non-finite points
    get rows of -1; lists are padded with -1 when the cloud has fewer than k finite points.  n x k int32."""
    pts = np.ascontiguousarray(pts, dtype=np.float32)
    out = np.full((len(pts), k), -1, dtype=np.int32)
    fi = np.flatnonzero(_finite(pts))
    m = len(fi)
    if m == 0:
        return out
    kk = min(k, m)
    f = pts[fi, :3]
    ids = fi.astype(np.uint64)[None, :]
    rows = max(1, (1 << 23) // m)          # about 8M distances per chunk
    for s in range(0, m, rows):
        q = f[s:s + rows]
        dx = q[:, 0:1] - f[None, :, 0]
        dy = q[:, 1:2] - f[None, :, 1]
        dz = q[:, 2:3] - f[None, :, 2]
        d2 = (dx * dx + dy * dy) + dz * dz
        # d2 >= 0, so its bits order like its value: one uint64 key orders by (d2, index)
        key = (d2.view(np.uint32).astype(np.uint64) << np.uint64(32)) | ids
        if kk < m:
            key = np.partition(key, kk - 1, axis=1)[:, :kk]
        key.sort(axis=1)
        out[fi[s:s + rows], :kk] = (key & np.uint64(0xFFFFFFFF)).astype(np.int32)
    return out


def normals_reference(pts, nbr, vp=(0.0, 0.0, 0.0), rows=None):
    """float64 normals over the given lists (-1 entries ignored): two-pass covariance, numpy eigh.  Returns a dict of
    normal (n x 3, unit, oriented towards vp where that is decided), curv = l0 / (l0 + l1 + l2), tol = angle tolerance
    2e-7 + 1e-13 l2 / (l1 - l0) (the float32 rounding of the output plus a double eigen-solve's error over the eigen-gap;
    inf where l1 == l0 leaves the normal undefined), signed = |n.(vp - p)| > 1e-9 |vp - p| (the orientation is decided),
    valid = at least 3 neighbours (otherwise the kernel writes NaN), and the eigenvalues w.  rows: the point each list
    belongs to (default: list i is point i's)."""
    P = pts[:, :3].astype(np.float64)
    n = len(nbr)
    rows_of = np.arange(n) if rows is None else np.asarray(rows)
    have = nbr >= 0
    cnt = have.sum(axis=1)
    valid = cnt >= 3
    res = dict(normal=np.full((n, 3), np.nan), curv=np.full(n, np.nan), tol=np.full(n, np.inf), signed=np.zeros(n, bool),
               valid=valid, w=np.full((n, 3), np.nan))
    todo = np.flatnonzero(valid)
    for s in range(0, len(todo), 200_000):
        r = todo[s:s + 200_000]
        h = have[r][:, :, None]
        X = P[np.where(have[r], nbr[r], 0)]
        c = (X * h).sum(axis=1) / cnt[r][:, None]
        D = (X - c[:, None, :]) * h
        C = np.einsum("nki,nkj->nij", D, D) / cnt[r][:, None, None]
        w, V = np.linalg.eigh(C)
        nv = V[:, :, 0]
        v = np.asarray(vp, dtype=np.float64)[None, :] - P[rows_of[r]]
        dot = (nv * v).sum(axis=1)
        nv = np.where(dot[:, None] < 0, -nv, nv)
        tr = w.sum(axis=1)
        with np.errstate(divide="ignore", invalid="ignore"):
            res["curv"][r] = np.where(tr > 0, np.abs(w[:, 0]) / tr, 0.0)
            gap = w[:, 1] - w[:, 0]
            res["tol"][r] = np.where(gap > 0, 2e-7 + 1e-13 * np.abs(w[:, 2]) / gap, np.inf)
        res["normal"][r] = nv
        res["signed"][r] = np.abs(dot) > 1e-9 * np.linalg.norm(v, axis=1)
        res["w"][r] = w
    return res


def normal_angles(got, ref):
    """Angle between the kernel's normals and the reference's: towards the oriented reference where the orientation is
    decided, to the nearer of +-reference elsewhere."""
    a = got[:, :3].astype(np.float64)
    b = ref["normal"]
    cross = np.linalg.norm(np.cross(a, b), axis=1)
    dot = (a * b).sum(axis=1)
    return np.arctan2(cross, np.where(ref["signed"], dot, np.abs(dot)))


def components_reference(pts, thr, seg):
    """mvr_denoise restated: components of the graph joining finite points with sqrt((double)dx^2 + dy^2 + dz^2) <= thr
    (the kernel's own predicate, in its own order of operations; candidate pairs from cKDTree with a relative 1e-9 slack),
    non-finite points singletons; components smaller than seg dropped; kept points ordered by their component's smallest
    index, then by index.  Returns (kept indices int32, noise count)."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    from scipy.spatial import cKDTree
    p = np.asarray(pts)[:, :3].astype(np.float64)
    n = len(p)
    ok = np.isfinite(p).all(axis=1)
    idx = np.flatnonzero(ok)
    pairs = cKDTree(p[ok]).query_pairs(thr * (1 + 1e-9), output_type="ndarray") if len(idx) else np.zeros((0, 2), np.int64)
    a, b = idx[pairs[:, 0]], idx[pairs[:, 1]]
    d = p[a] - p[b]
    e = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]) <= thr
    g = coo_matrix((np.ones(int(e.sum()), dtype=np.int8), (a[e], b[e])), shape=(n, n))
    _, label = connected_components(g, directed=False)
    size = np.bincount(label)
    first = np.full(len(size), n, dtype=np.int64)
    np.minimum.at(first, label, np.arange(n))
    keep = np.flatnonzero(size[label] >= seg)
    order = np.lexsort((keep, first[label[keep]]))
    return keep[order].astype(np.int32), int(n - len(keep))


def pair_grid_shape(pts, e):
    """make_pair_grid's sizing (csrc/api.cu, isotropic cells): ([nx, ny, nz], final cell edge) for the finite points'
    bounding box and requested edge e -- each axis capped at 4096 cells, the edge grown by 1.25 until the table fits."""
    f = pts[_finite(pts), :3]
    ext = f.max(axis=0).astype(np.float64) - f.min(axis=0).astype(np.float64)
    while True:
        n = [int(min(4096.0, np.floor(x / e) + 3.0)) for x in ext]
        if n[0] * n[1] * n[2] <= MAX_CELLS:
            return n, e
        e *= 1.25


# ---- clouds -----------------------------------------------------------------------------------------------------------
def _xyz1(p):
    out = np.ones((len(p), 4), dtype=np.float32)
    out[:, :3] = p
    return out


def _poison(pts, every, start=0):
    """Every `every`-th point from `start` made non-finite: NaN x, +inf y, -inf z in turn."""
    pts = pts.copy()
    for j, i in enumerate(range(start, len(pts), every)):
        pts[i, j % 3] = (np.nan, np.inf, -np.inf)[j % 3]
    return pts


def _interleave(base, extra, seed):
    """base and extra concatenated, then the extra points moved to seeded positions among the base points."""
    pts = np.concatenate([base, extra])
    return pts[np.random.default_rng(seed).permutation(len(pts))]


def _view(synth, n=12_000):
    v, _ = synth.turntable_view(3, 12, n)
    return v


def normals_cloud(case, synth):
    """(points, viewpoint, cell_edge option (0: the default grid), collinear line (ids, unit direction) or None)."""
    vp0 = (0.0, 0.0, 0.0)
    if case == "view":                      # a partial view with non-finite points, default grid
        return _poison(_view(synth), 97, 5), (10.0, -20.0, 30.0), 0.0, None
    if case == "tiny_cell":                 # the same view binned in grown tiny cells: many shells per point
        return _poison(_view(synth), 97, 5), vp0, 0.01, None
    if case == "huge_cell":                 # ... and in one single cell
        return _poison(_view(synth), 97, 5), vp0, 1.0e4, None
    if case == "outliers":                  # isolated points tens of cells from everything, a 5-point cluster far away
        v = _poison(_view(synth), 97, 5)
        rng = np.random.default_rng(3)
        d = rng.normal(size=(20, 3))
        far = np.asarray(synth.CENTER) + d / np.linalg.norm(d, axis=1, keepdims=True) * rng.uniform(140, 260, (20, 1))
        cluster = np.array([250.0, -180.0, 700.0]) + rng.normal(size=(5, 3)) * 0.3
        return _interleave(v, _xyz1(np.concatenate([far, cluster])), 4), vp0, 0.0, None
    if case == "duplicates":                # stacks of 40 identical points, 5 copies of one surface point
        v = _view(synth, 6_000)
        on_surface = np.repeat(v[100:101], 40, axis=0)
        off_surface = np.repeat(_xyz1(np.array([[0.0, 150.0, 900.0]])), 40, axis=0)
        five = np.repeat(v[2000:2001], 5, axis=0)
        return _interleave(v, np.concatenate([on_surface, off_surface, five]), 5), vp0, 0.0, None
    if case == "flat":                      # zero extent in z (exactly 900): a square lattice, three cells deep in z
        i, j = np.meshgrid(np.arange(60), np.arange(60), indexing="ij")
        p = np.stack([-15.0 + 0.5 * i.ravel(), 20.0 + 0.5 * j.ravel(), np.full(i.size, 900.0)], axis=1)
        return _interleave(_xyz1(p), np.zeros((0, 4), np.float32), 6), vp0, 0.0, None
    if case == "thin_capped":               # 1000 mm long, 0.1 mm cells: the x axis is capped at 4096 cells
        rng = np.random.default_rng(7)
        p = np.stack([rng.uniform(0, 1000, 8000), rng.uniform(-1, 1, 8000), 900 + rng.uniform(-1, 1, 8000)], axis=1)
        return _xyz1(p), vp0, 0.1, None
    if case == "far":                       # a 1 mm bumpy sphere at (1e4, -1e4, 5e3), 0.05 mm spacing, viewed from its centre
        o = np.array([1.0e4, -1.0e4, 5.0e3])
        p = (synth.full_object(5_000, seed=9)[:, :3].astype(np.float64) - synth.CENTER) / 100.0 + o
        return _xyz1(p), tuple(o), 0.0, None
    if case == "degenerate":                # an exactly collinear run, an isolated stack, a 3 x 3 x 3 cube lattice
        t = 0.25 * np.arange(200)
        line = np.stack([900.0 + t, -50.0 + 2.0 * t, 30.0 - t], axis=1)
        stack = np.repeat([[-300.0, 40.0, 500.0]], 40, axis=0)
        g = np.stack(np.meshgrid(*[np.arange(3.0)] * 3, indexing="ij"), axis=-1).reshape(-1, 3) * 0.5 + [300.0, 300.0, 300.0]
        pts = _xyz1(np.concatenate([line, stack, g]))
        perm = np.random.default_rng(8).permutation(len(pts))
        pts = pts[perm]
        line_ids = np.flatnonzero(perm < 200)
        return pts, vp0, 0.0, (line_ids, np.array([1.0, 2.0, -1.0]) / np.sqrt(6.0))
    raise KeyError(case)


SAME_POINTS = {"tiny_cell": "view", "huge_cell": "view"}   # cases that bin the same points in another grid
NORMAL_CASES = ["view", "outliers", "duplicates", "flat", "thin_capped", "tiny_cell", "huge_cell", "far", "degenerate"]

_cache = {}


def _cached(key, fn):
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


def check_normals(pts, nbr, nrm, vp, line=None, rows=None):
    """The kernel's normals / curvatures (nrm, n x 4) on its own lists (nbr) against normals_reference, plus the exact
    expectations of degenerate neighbourhoods.  rows: the points nbr / nrm belong to (default: all, in order)."""
    rows_of = np.arange(len(nbr)) if rows is None else np.asarray(rows)
    ref = normals_reference(pts, nbr, vp, rows_of)
    v = ref["valid"]
    assert np.isnan(nrm[~v]).all(), "fewer than 3 neighbours must give NaN"
    assert np.isfinite(nrm[v]).all()
    got = nrm[v]
    assert np.all(np.abs(np.linalg.norm(got[:, :3].astype(np.float64), axis=1) - 1.0) <= 1e-6)
    sub = {key: val[v] for key, val in ref.items()}
    ang = normal_angles(got, sub)
    bad = ang > sub["tol"]
    assert not bad.any(), "%d normals off: worst %g rad (tolerance %g)" % (bad.sum(), ang[bad].max(), sub["tol"][bad][np.argmax(ang[bad])])
    dc = np.abs(got[:, 3].astype(np.float64) - sub["curv"])
    cbad = dc > 2e-7 * sub["curv"] + 1e-12
    assert not cbad.any(), "%d curvatures off: worst %g" % (cbad.sum(), dc.max())
    # orientation: towards the viewpoint wherever that is decided
    P = pts[rows_of[v], :3].astype(np.float64)
    s = (got[:, :3].astype(np.float64) * (np.asarray(vp, dtype=np.float64) - P)).sum(axis=1)
    assert np.all(s[sub["signed"]] > 0)
    # exact cases, found from the lists themselves
    nb = nbr[v]
    X = pts[np.where(nb >= 0, nb, nb[:, :1]), :3]
    same = (X == X[:, :1]).all(axis=1)                     # per coordinate: every neighbour equal to the first
    ident = same.all(axis=1)
    if ident.any():                                       # all identical: a unit axis vector, curvature exactly 0
        a = np.abs(got[ident, :3])
        assert np.all((np.sort(a, axis=1) == [0.0, 0.0, 1.0]).all(axis=1)) and np.all(got[ident, 3] == 0.0)
    xy = X[:, :, :2].astype(np.float64)
    xy = xy - xy.mean(axis=1, keepdims=True)
    cxy = np.einsum("nki,nkj->nij", xy, xy)
    planar = same[:, 2] & (np.linalg.det(cxy) > 1e-12 * np.einsum("nii->n", cxy) ** 2)
    if planar.any():                                      # z constant, spread in x and y: (0, 0, +-1) exactly, curvature 0
        g = got[planar]
        assert np.all(g[:, 0] == 0.0) and np.all(g[:, 1] == 0.0) and np.all(np.abs(g[:, 2]) == 1.0) and np.all(g[:, 3] == 0.0)
    if line is not None:                                  # exactly collinear lists: orthogonal to the line, curvature ~0
        ids, u = line
        on = np.isin(nbr, ids) | (nbr < 0)
        col = v & on.all(axis=1) & np.isin(rows_of, ids)
        assert col.sum() >= 150
        g = nrm[col, :3].astype(np.float64)
        assert np.all(np.abs(g @ u) <= 1e-6) and np.all(nrm[col, 3] <= 1e-12)
    return ref


# ---- CPU self-checks of the references --------------------------------------------------------------------------------
def _tie_cloud():
    """A lattice (many equal distances), duplicates and non-finite points."""
    g = np.stack(np.meshgrid(np.arange(8.0), np.arange(8.0), np.arange(2.0), indexing="ij"), axis=-1).reshape(-1, 3)
    p = _xyz1(np.concatenate([g * 0.5 + 900.0, np.repeat(g[5:6] * 0.5 + 900.0, 6, axis=0), [[950.0, 950.0, 950.0]]]))
    p = p[np.random.default_rng(1).permutation(len(p))]
    return _poison(p, 17, 3)


@pytest.mark.parametrize("k", [3, 16, 17, 32])
def test_knn_reference_equals_the_oracle_on_ties_and_duplicates(orc, synth, k):
    for pts in (_tie_cloud(), _poison(synth.full_object(3000, seed=2, noise=0.1), 41, 1), _tie_cloud()[:k - 1]):
        _, onbr = orc.estimate_normals(pts, k, want_neighbours=True)
        assert np.array_equal(knn_reference(pts, k), onbr)


def test_knn_reference_pads_short_lists_and_orders_ties_by_index():
    pts = _xyz1(np.array([[0.0, 0, 0], [1.0, 0, 0], [0.0, 0, 0], [-1.0, 0, 0], [np.nan, 0, 0]]))
    got = knn_reference(pts, 6)
    assert got[0].tolist() == [0, 2, 1, 3, -1, -1]
    assert got[2].tolist() == [0, 2, 1, 3, -1, -1]
    assert got[1].tolist() == [1, 0, 2, 3, -1, -1]
    assert got[4].tolist() == [-1] * 6


def test_normals_reference_on_hand_built_neighbourhoods():
    rng = np.random.default_rng(4)
    # a tilted plane: the normal is known, the curvature 0
    nrm = np.array([1.0, -2.0, 2.0]) / 3.0
    u = np.array([2.0, 2.0, 1.0]) / 3.0
    w = np.cross(nrm, u)
    ab = rng.uniform(-1, 1, (12, 2))
    plane = np.array([5.0, 5.0, 5.0]) + ab[:, :1] * u + ab[:, 1:] * w
    # an anisotropic blob along the axes: smallest spread along y
    blob = rng.normal(size=(16, 3)) * [3.0, 0.1, 1.0] + [0.0, 0.0, -40.0]
    line = np.outer(np.arange(6.0), [1.0, 1.0, 0.0])
    pts = _xyz1(np.concatenate([plane, blob, line, np.zeros((4, 3)) + 7.0]))
    nbr = np.full((len(pts), 16), -1, dtype=np.int32)
    nbr[0, :12] = np.arange(12)
    nbr[1, :16] = 12 + np.arange(16)
    nbr[2, :6] = 28 + np.arange(6)
    nbr[3, :4] = 34 + np.arange(4)
    nbr[4, :2] = [0, 1]
    ref = normals_reference(pts, nbr, vp=(0.0, 0.0, 0.0))
    assert abs(abs(ref["normal"][0] @ nrm) - 1) < 1e-12 and ref["curv"][0] < 1e-12 and ref["tol"][0] < 1e-6
    assert ref["normal"][0] @ (-pts[0, :3]) > 0                       # oriented towards the viewpoint
    assert abs(abs(ref["normal"][1][1]) - 1) < 1e-3 and ref["signed"][1]
    assert ref["tol"][2] > 1e-3 and ref["curv"][2] < 1e-12             # collinear: the normal is not defined
    assert ref["curv"][3] == 0.0 and np.isinf(ref["tol"][3])         # identical
    assert not ref["valid"][4] and np.isnan(ref["curv"][4])
    got = np.empty((len(pts), 4), np.float32)
    got[:, :3], got[:, 3] = ref["normal"], ref["curv"]
    a = normal_angles(got, ref)
    assert np.all(a[:2] < 1e-7)


def _specks_cloud(synth):
    rng = np.random.default_rng(21)
    scan, _ = synth.turntable_view(2, 12, 8_000)
    c = rng.uniform(-80, 80, (30, 3)) + [0, 0, 1000]
    specks = np.concatenate([cc + rng.normal(size=(1 + k % 12, 3)) * 0.4 for k, cc in enumerate(c)])
    pts = np.concatenate([scan, _xyz1(specks)])
    return pts[rng.permutation(len(pts))]


def test_components_reference_equals_the_oracle(orc, synth):
    pts = _specks_cloud(synth)
    for seg, thr in ((10, 2.5), (3, 1.0), (1, 0.5), (0, 2.0)):
        (keep, noise), (okeep, onoise) = components_reference(pts, thr, seg), orc.denoise(pts, seg, thr)
        assert noise == onoise and np.array_equal(keep, okeep)


def test_denoise_cases_reach_their_edges():
    """The data of the GPU cases does what it is meant to: edges at exactly the threshold and none one ulp beyond, the cut
    helix has its 8 components and orders them differently by smallest and by largest index (a union-find whose roots are
    not the smallest index is visible), and the grids are grown or capped."""
    p, thr = lattice(0.5)
    assert len(components_reference(p, thr, len(p))[0]) == len(p)
    q, _ = lattice(np.float32(0.5) + np.float32(2.0 ** -14))
    assert len(components_reference(q, thr, 2)[0]) == 0
    pts, sizes, label = helix(cuts=HELIX_CUTS)
    keep, _ = components_reference(pts, 1.0, 1)
    starts = np.r_[0, np.flatnonzero(np.diff(label[keep]) != 0) + 1]
    assert len(starts) == 8 and np.diff(np.r_[starts, len(keep)]).tolist() == [sizes[c] for c in label[keep][starts]]
    lo = [np.flatnonzero(label == c).min() for c in range(8)]
    hi = [np.flatnonzero(label == c).max() for c in range(8)]
    assert np.argsort(lo).tolist() != np.argsort(hi).tolist()
    assert pair_grid_shape(pts, 1.0 * 1.0001)[1] > 1.0001
    line = long_line()
    assert pair_grid_shape(line, 1.0001)[0][0] == 4096 and (line[:, 0] - line[:, 0].min()).max() > 4096 * 1.0001


# ---- denoise data -----------------------------------------------------------------------------------------------------
def lattice(spacing, m=24):
    """m^3 lattice at offset 900 spaced `spacing` (float32-exact coordinates), shuffled; threshold 0.5."""
    i = np.stack(np.meshgrid(*[np.arange(m, dtype=np.float32)] * 3, indexing="ij"), axis=-1).reshape(-1, 3)
    p = _xyz1(np.float32(900.0) + i * np.float32(spacing))
    return p[np.random.default_rng(11).permutation(len(p))], 0.5


HELIX_CUTS = [1000, 1010, 50_000, 80_000, 80_012, 120_000, 170_000]   # removed points: segments of 9 and 11 among them


def helix(n=200_000, step=0.9, radius=50.0, pitch=3.0, cuts=()):
    """A helix of n points `step` apart along the curve (threshold 1: only consecutive points are joined), the points at
    positions `cuts` removed, shuffled.  Returns (points, segment sizes, segment label of every output point)."""
    turn = np.hypot(2 * np.pi * radius, pitch)
    t = np.arange(n) * step / turn * 2 * np.pi
    p = np.stack([radius * np.cos(t), radius * np.sin(t), 900.0 + pitch * t / (2 * np.pi)], axis=1)
    keep = np.ones(n, bool)
    keep[list(cuts)] = False
    seg = np.cumsum(~keep)[keep]
    pts = _xyz1(p[keep])
    perm = np.random.default_rng(12).permutation(len(pts))
    return pts[perm], np.bincount(seg).tolist(), seg[perm]


def long_line(n=6_000, step=0.9):
    """A 5.4 m line along x (threshold 1): its grid axis is capped at 4096 cells, the far points share the last cell."""
    x = np.arange(n) * step
    return _xyz1(np.stack([x - 2000.0, 0.1 * np.sin(x), np.full(n, 900.0)], axis=1))


def sized_clusters(sizes, seed, apart=20.0):
    """Tight chains (0.5 mm steps) of the given sizes `apart` mm apart, shuffled; threshold 1."""
    parts = []
    for j, s in enumerate(sizes):
        o = np.array([apart * (j % 10), 20.0 * (j // 10), 900.0])
        parts.append(o + np.outer(np.arange(s) * 0.5, [0.6, 0.0, 0.8]))
    p = _xyz1(np.concatenate(parts))
    return p[np.random.default_rng(seed).permutation(len(p))]


# ---- GPU: neighbour lists and normals ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def nctx(mvr):
    c = mvr.Context(0)   # raises without a CUDA device: there is no fallback
    yield c
    c.close()


def gpu_normals(c, mvr, which, pts, k, vp=(0.0, 0.0, 0.0), cell_edge=0.0):
    """mvr_estimate_normals on slot `which`, with the index options set for this call and reset after it."""
    c.set_index_options(cell_edge=cell_edge)
    try:
        (c.set_source if which == mvr.SOURCE else c.set_target)(pts)
        return c.estimate_normals(which, len(pts), k, viewpoint=vp, want_neighbours=True)
    finally:
        c.set_index_options(cell_edge=0.0)


def _case(case, synth):
    pts, vp, ce, line = _cached(("cloud", case), lambda: normals_cloud(case, synth))
    ref = _cached(("knn", SAME_POINTS.get(case, case)), lambda: knn_reference(pts, 32))
    return pts, vp, ce, line, ref


def _grid_of(case, pts, ce):
    if case == "thin_capped":
        assert pair_grid_shape(pts, float(np.float32(ce)))[0][0] == 4096
        assert (pts[:, 0].max() - pts[:, 0].min()) > 4096 * float(np.float32(ce)) * 2
    if case == "tiny_cell":
        assert pair_grid_shape(pts, float(np.float32(ce)))[1] > 50 * ce
    if case == "huge_cell":
        assert pair_grid_shape(pts, float(np.float32(ce)))[0] == [3, 3, 3]
    if case == "flat":
        assert np.ptp(pts[:, 2]) == 0


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("case", NORMAL_CASES)
def test_neighbour_lists_bit_exact(nctx, mvr, synth, case, k):
    pts, vp, ce, _, ref = _case(case, synth)
    _grid_of(case, pts, ce)
    for which in (mvr.SOURCE, mvr.TARGET):
        _, nbr = gpu_normals(nctx, mvr, which, pts, k, vp, ce)
        bad = np.flatnonzero((nbr != ref[:, :k]).any(axis=1))
        assert len(bad) == 0, "%d lists differ, first at point %d: %s vs %s" % (len(bad), bad[0], nbr[bad[0]], ref[bad[0], :k])


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("case", NORMAL_CASES)
def test_normals_match_float64_reference(nctx, mvr, synth, case, k):
    pts, vp, ce, line, _ = _case(case, synth)
    for which in (mvr.SOURCE, mvr.TARGET):
        nrm, nbr = gpu_normals(nctx, mvr, which, pts, k, vp, ce)
        ref = check_normals(pts, nbr, nrm, vp, line)
        if case == "flat" and k >= 7:   # every list spans the plane: (0, 0, -1) towards the origin, curvature 0
            assert np.all(nrm[:, :3] == [0.0, 0.0, -1.0]) and np.all(nrm[:, 3] == 0.0)
        if case == "far":               # viewed from the sphere's centre: the orientation is decided (and checked) nearly everywhere
            assert ref["signed"].mean() > 0.95


@pytest.mark.gpu
@pytest.mark.parametrize("k", KS)
def test_short_clouds(nctx, mvr, k):
    """n = 2, 3, k - 1, k, k + 1 finite points (and one NaN): lists padded with -1, NaN normals below 3 neighbours."""
    for n in sorted({2, 3, k - 1, k, k + 1} - {1}):
        rng = np.random.default_rng(100 + n)
        pts = _xyz1(rng.normal(size=(n + 1, 3)) * 2.0 + [0.0, 0.0, 900.0])
        pts[n // 2, 0] = np.nan
        ref = knn_reference(pts, k)
        for which in (mvr.SOURCE, mvr.TARGET):
            nrm, nbr = gpu_normals(nctx, mvr, which, pts, k)
            assert np.array_equal(nbr, ref), "n = %d" % n
            check_normals(pts, nbr, nrm, (0.0, 0.0, 0.0))
            if n == 2:
                assert np.isnan(nrm).all() and (nbr[:, 2:] == -1).all()


@pytest.mark.gpu
def test_two_million_points_k32_against_the_kdtree(nctx, mvr, orc, synth):
    pts = _poison(synth.full_object(2_000_000, seed=7, noise=0.05), 9973, 17)
    _, onbr = orc.estimate_normals(pts, 32, want_neighbours=True)
    nrm, nbr = gpu_normals(nctx, mvr, mvr.TARGET, pts, 32)
    assert np.array_equal(nbr, onbr)
    sel = np.arange(0, len(pts), 16)
    check_normals(pts, nbr[sel], nrm[sel], (0.0, 0.0, 0.0), rows=sel)


# ---- GPU: denoise -----------------------------------------------------------------------------------------------------
def run_denoise(c, pts, seg, thr):
    """The kernel's (kept, noise) against components_reference; a second call must give the same output."""
    keep, noise = c.denoise(pts, seg, thr)
    want, wnoise = components_reference(pts, thr, seg)
    assert noise == wnoise and len(keep) + noise == len(pts)
    assert np.array_equal(keep, want)
    keep2, noise2 = c.denoise(pts, seg, thr)
    assert noise2 == noise and np.array_equal(keep2, keep)
    return keep, noise


@pytest.mark.gpu
def test_denoise_edges_at_exactly_the_threshold(nctx):
    p, thr = lattice(0.5)
    keep, noise = run_denoise(nctx, p, 10, thr)
    assert noise == 0 and np.array_equal(keep, np.arange(len(p)))           # one component
    q, _ = lattice(np.float32(0.5) + np.float32(2.0 ** -14))                 # one float ulp (at 900) wider: no edge at all
    keep, noise = run_denoise(nctx, q, 2, thr)
    assert len(keep) == 0 and noise == len(q)
    keep, noise = run_denoise(nctx, q, 1, thr)
    assert noise == 0 and np.array_equal(keep, np.arange(len(q)))


@pytest.mark.gpu
def test_denoise_long_chains(nctx):
    pts, _, _ = helix()
    keep, noise = run_denoise(nctx, pts, 10, 1.0)                             # 200k points, one path
    assert noise == 0 and np.array_equal(keep, np.arange(len(pts)))
    pts, sizes, label = helix(cuts=HELIX_CUTS)
    keep, noise = run_denoise(nctx, pts, 1, 1.0)                              # cut at 7 places: 8 components
    starts = np.r_[0, np.flatnonzero(np.diff(label[keep]) != 0) + 1]
    assert len(starts) == 8 and sorted(np.diff(np.r_[starts, len(keep)]).tolist()) == sorted(sizes)
    keep, noise = run_denoise(nctx, pts, 10, 1.0)                             # the 9-point piece is noise
    assert noise == 9


@pytest.mark.gpu
def test_denoise_two_million_points_one_component_plus_specks(nctx, synth):
    u = synth._directions(13, np.arange(2_000_000, dtype=np.uint64))
    obj = _xyz1(synth.CENTER + 100.0 * u)                                   # a ball: about 32 points within 0.8 mm of each
    rng = np.random.default_rng(14)
    c = rng.uniform(-1, 1, (40, 3))
    c = synth.CENTER + 160.0 * c / np.linalg.norm(c, axis=1, keepdims=True)
    specks = _xyz1(np.concatenate([cc + rng.normal(size=(1 + j % 12, 3)) * 0.2 for j, cc in enumerate(c)]))
    pts = _interleave(obj, specks, 15)
    keep, noise = run_denoise(nctx, pts, 20, 0.8)
    assert len(keep) >= 2_000_000 and noise == len(specks)


@pytest.mark.gpu
def test_denoise_segment_threshold_boundary(nctx):
    sizes = [9, 10, 11] * 20
    pts = sized_clusters(sizes, 16)
    keep, noise = run_denoise(nctx, pts, 10, 1.0)
    assert noise == 9 * 20 and len(keep) == 21 * 20
    keep, noise = run_denoise(nctx, pts, 11, 1.0)
    assert noise == 19 * 20


@pytest.mark.gpu
def test_denoise_cells_full_of_duplicates(nctx):
    pts = _xyz1(np.concatenate([np.repeat([[1.0, 2.0, 900.0]], 5000, axis=0), np.repeat([[40.0, 2.0, 900.0]], 3, axis=0),
                                [[1.5, 2.0, 900.0], [41.0, 2.0, 900.0]]]))
    pts = pts[np.random.default_rng(17).permutation(len(pts))]
    keep, noise = run_denoise(nctx, pts, 10, 1.0)
    assert len(keep) == 5001 and noise == 4


@pytest.mark.gpu
@pytest.mark.parametrize("seg", [0, 1, 3])
def test_denoise_non_finite_points(nctx, synth, seg):
    pts = _poison(_specks_cloud(synth), 7, 2)
    run_denoise(nctx, pts, seg, 2.5)


@pytest.mark.gpu
def test_denoise_capped_grids(nctx, synth):
    obj = synth.full_object(300_000, seed=18)
    assert pair_grid_shape(obj, 0.3 * 1.0001)[1] > 2 * 0.3            # the cells grow to fit the table
    run_denoise(nctx, obj, 10, 0.3)
    line = long_line()
    run_denoise(nctx, line, 10, 1.0)                                  # an axis capped at 4096 cells
    pts = sized_clusters([9, 10, 11, 40], 19, apart=1500.0)         # clusters in the capped cells, far from the line
    run_denoise(nctx, np.concatenate([line, pts]), 10, 1.0)
