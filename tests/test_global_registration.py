"""Global registration without an initial guess: FPFH features of index-strided keypoints on the GPU, exact mutual feature
matches, seeded RANSAC hypotheses with edge pre-rejection, scored by the GPU scorer (mvr_compute_fpfh, mvr_match_features,
mvr_global_align).  The features and the matcher are compared with a numpy restatement; the pipeline with seeded arbitrary
placements of the object."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EDGE_TOL = 1e-9


def rot_angle(A, B):
    R = np.asarray(A, dtype=np.float64)[:3, :3] @ np.asarray(B, dtype=np.float64)[:3, :3].T
    return float(np.arccos(np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0)))


def centre_error(A, B, c):
    c = np.append(np.asarray(c, dtype=np.float64), 1.0)
    return float(np.linalg.norm((np.asarray(A, dtype=np.float64) @ c - np.asarray(B, dtype=np.float64) @ c)[:3]))


# ---- the features, restated in numpy (double, the kernels' operation order) ---------------------------------------------
def pair_features(p1, n1, p2, n2):
    """pcl::computePairFeatures on float32 inputs (..., 3) in float64: (f1, f2, f3, ok)."""
    p1, n1, p2, n2 = (np.asarray(a, dtype=np.float32).astype(np.float64) for a in (p1, n1, p2, n2))
    d = p2 - p1
    f4 = np.sqrt((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2])
    ok = f4 != 0
    f4s = np.where(ok, f4, 1.0)
    dot = lambda a, b: (a[..., 0] * b[..., 0] + a[..., 1] * b[..., 1]) + a[..., 2] * b[..., 2]
    a1, a2 = dot(n1, d) / f4s, dot(n2, d) / f4s
    sw = np.abs(a1) < np.abs(a2)
    N1 = np.where(sw[..., None], n2, n1)
    N2 = np.where(sw[..., None], n1, n2)
    d = np.where(sw[..., None], -d, d)
    f3 = np.where(sw, -a2, a1)
    cross = lambda a, b: np.stack([a[..., 1] * b[..., 2] - a[..., 2] * b[..., 1], a[..., 2] * b[..., 0] - a[..., 0] * b[..., 2],
                                   a[..., 0] * b[..., 1] - a[..., 1] * b[..., 0]], axis=-1)
    v = cross(d, N1)
    vn = np.sqrt((v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1]) + v[..., 2] * v[..., 2])
    ok = ok & (vn != 0)
    v = v / np.where(vn != 0, vn, 1.0)[..., None]
    w = cross(N1, v)
    f2 = dot(v, N2)
    f1 = np.arctan2(dot(w, N2), dot(N1, N2))
    return f1, f2, f3, ok


def bin_values(f1, f2, f3):
    """The unfloored bin coordinates 11 (f + offset) / range of the three features."""
    return 11.0 * (f1 + np.pi) / (2.0 * np.pi), 11.0 * (f2 + 1.0) / 2.0, 11.0 * (f3 + 1.0) / 2.0


def bins_of(t):
    return np.clip(np.floor(t), 0, 10).astype(np.int64)


def near_edge(t):
    r = np.round(t)
    return (np.abs(t - r) < EDGE_TOL) & (r >= 1) & (r <= 10)


def taken_lists(nbr, k):
    """Which list entries a keypoint's features use: the first k - 1 that are neither -1 nor itself."""
    n = len(nbr)
    m = (nbr >= 0) & (nbr != np.arange(n)[:, None])
    return m & (np.cumsum(m, axis=1) <= k - 1)


def d2_pinned(q, t):
    d = (np.asarray(q, dtype=np.float32) - np.asarray(t, dtype=np.float32)).astype(np.float32)
    return ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]).astype(np.float32)


def fpfh_numpy(kp, nrm, nbr, k):
    """(descriptors n x 33 float32, keypoints with a pair feature within EDGE_TOL of a bin edge)."""
    kp = np.asarray(kp, dtype=np.float32)[:, :3]
    nv = np.asarray(nrm, dtype=np.float32)[:, :3]
    n = len(kp)
    fin = np.isfinite(nv).all(axis=1)
    take = taken_lists(nbr, k)
    cnt = np.zeros((n, 33), dtype=np.int64)
    edge = np.zeros(n, dtype=bool)
    for a in range(nbr.shape[1]):
        j = np.where(take[:, a], nbr[:, a], 0)
        use = take[:, a] & fin & fin[j]
        rows = np.nonzero(use)[0]
        f1, f2, f3, ok = pair_features(kp[rows], nv[rows], kp[j[rows]], nv[j[rows]])
        rows = rows[ok]
        for off, t in zip((0, 11, 22), bin_values(f1[ok], f2[ok], f3[ok])):
            np.add.at(cnt, (rows, off + bins_of(t)), 1)
            edge[rows[near_edge(t)]] = True
    inc = 100.0 / (k - 1)
    seq = np.zeros(k + 1)
    for c in range(1, k + 1):
        seq[c] = seq[c - 1] + inc
    spfh = seq[cnt]
    acc = np.zeros((n, 33))
    for a in range(nbr.shape[1]):
        j = np.where(take[:, a], nbr[:, a], 0)
        d2 = d2_pinned(kp, kp[j])
        use = take[:, a] & (d2 != 0)
        w = 1.0 / np.where(use, d2, 1).astype(np.float64)
        acc[use] = acc[use] + spfh[j[use]] * w[use, None]
    out = np.empty((n, 33), dtype=np.float32)
    for s in range(3):
        sub = slice(11 * s, 11 * s + 11)
        tot = np.zeros(n)
        for b in range(11 * s, 11 * s + 11):
            tot = tot + acc[:, b]
        scale = np.where(tot != 0, 100.0 / np.where(tot != 0, tot, 1.0), 0.0)
        out[:, sub] = (spfh[:, sub] + acc[:, sub] * scale[:, None]).astype(np.float32)
    out[~fin] = 0
    return out, edge


def match_numpy(a, b):
    """Exact nearest row of b for every row of a: squared L2 summed in bin order in float32, ties to the lowest row, all-zero rows
    never match."""
    a = np.asarray(a, dtype=np.float32)
    b = np.asarray(b, dtype=np.float32)
    out = np.full(len(a), -1, dtype=np.int32)
    if len(b) == 0:
        return out
    bz = ~(b != 0).any(axis=1)
    for i0 in range(0, len(a), 256):
        q = a[i0:i0 + 256]
        d = np.zeros((len(q), len(b)), dtype=np.float32)
        for c in range(33):
            t = (q[:, None, c] - b[None, :, c]).astype(np.float32)
            d = (d + t * t).astype(np.float32)
        d[:, bz] = np.inf
        best = np.argmin(d, axis=1)   # the first minimum: the lowest row
        ok = np.isfinite(d[np.arange(len(q)), best]) & (q != 0).any(axis=1)
        out[i0:i0 + 256] = np.where(ok, best, -1)
    return out


def keypoint_index(pts, keypoints):
    n = len(pts)
    stride = max(1, -(-n // keypoints))
    i = np.arange(0, n, stride)
    return i[np.isfinite(pts[i, :3]).all(axis=1)]


# ---- the pipeline, restated with scipy (CPU) ------------------------------------------------------------------------------
def pipeline_numpy(src, tgt, seed, keypoints=4096, k=32, hypotheses=1000, samples=2048, max_dist=4.0):
    from scipy.spatial import cKDTree
    feats = []
    for P in (src, tgt):
        P = np.asarray(P, dtype=np.float32)
        kp = P[keypoint_index(P, keypoints), :3].astype(np.float64)
        d, nb = cKDTree(kp).query(kp, k=k)
        q = kp[nb]
        C = np.einsum("nki,nkj->nij", q - q.mean(1, keepdims=True), q - q.mean(1, keepdims=True)) / k
        nrm = np.linalg.eigh(C)[1][:, :, 0]
        vp = (P[:, :3].min(0).astype(np.float64) + P[:, :3].max(0)) * 0.5
        nrm[np.einsum("ni,ni->n", nrm, vp - kp) < 0] *= -1
        f, _ = fpfh_numpy(kp.astype(np.float32), nrm.astype(np.float32), nb.astype(np.int64), k)
        feats.append((kp, f))
    (ks, fs), (kt, ft) = feats
    st, ts = cKDTree(ft).query(fs)[1], cKDTree(fs).query(ft)[1]
    mut = np.nonzero(ts[st] == np.arange(len(fs)))[0]
    A, B = ks[mut], kt[st[mut]]
    rng = np.random.default_rng(seed)
    diag = np.linalg.norm(ks.max(0) - ks.min(0))
    hyps = []
    while len(hyps) < hypotheses:
        tri = np.stack([rng.choice(len(A), 3, replace=False) for _ in range(4096)])
        ea = np.linalg.norm(A[tri] - A[np.roll(tri, 1, axis=1)], axis=2)
        eb = np.linalg.norm(B[tri] - B[np.roll(tri, 1, axis=1)], axis=2)
        ok = (ea.min(1) >= 0.05 * diag) & ((np.minimum(ea, eb) / np.maximum(ea, eb)).min(1) >= 0.9)
        hyps.extend(tri[ok][: hypotheses - len(hyps)])
    tree = cKDTree(np.asarray(tgt, dtype=np.float64)[:, :3])
    samp = np.asarray(src, dtype=np.float64)[:: max(1, -(-len(src) // samples)), :3]
    best, pose = None, None
    for tri in hyps:
        a, b = A[tri], B[tri]
        H = (b - b.mean(0)).T @ (a - a.mean(0))
        U, _, Vt = np.linalg.svd(H)
        R = U @ np.diag([1, 1, np.sign(np.linalg.det(U @ Vt))]) @ Vt
        t = b.mean(0) - R @ a.mean(0)
        d, _ = tree.query(samp @ R.T + t, distance_upper_bound=max_dist)
        cost = np.where(np.isfinite(d), np.floor(d * d * (2 ** 24) / (max_dist * max_dist)), 2 ** 24).sum()
        if best is None or cost < best:
            best, pose = cost, np.eye(4)
            pose[:3, :3], pose[:3, 3] = R, t
    return pose, len(mut)


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_pair_features_on_hand_built_cases():
    n_up, n_x, n_t = np.array([0.0, 0.0, 1.0]), np.array([1.0, 0.0, 0.0]), np.array([0.6, 0.0, 0.8])
    p0, p1 = np.zeros(3), np.array([1.0, 0.0, 0.0])
    a = -float(np.float32(0.6))
    # |a1| = 0 < |a2| = 0.6: the roles swap, dp is negated and f3 = -a2
    f1, f2, f3, ok = pair_features(p0, n_up, p1, n_t)
    assert ok and f3 == a
    f1s, f2s, f3s, ok = pair_features(p1, n_t, p0, n_up)   # the same pair seen from the other end: no swap, f3 = a1
    assert ok and f3s == a and f1 == f1s and f2 == f2s
    # f4 == 0: skipped
    assert not pair_features(p0, n_up, p0, n_x)[3]
    # dp parallel to the first normal: |v| == 0, skipped
    assert not pair_features(p0, n_x, p1, n_x)[3]
    # coplanar normals: f1 = f2 = f3 = 0, every bin coordinate in the middle bin
    f1, f2, f3, ok = pair_features(p0, n_up, p1, n_up)
    assert ok and (f1, f2, f3) == (0.0, 0.0, 0.0)
    assert [int(bins_of(t)) for t in bin_values(f1, f2, f3)] == [5, 5, 5]
    # bin edges and clamping: f = -1 and f = +1 land in bins 0 and 10, f1 = +-pi too
    t1, t2, t3 = bin_values(np.array([-np.pi, np.pi]), np.array([-1.0, 1.0]), np.array([-1.0 - 1e-12, 1.0 + 1e-12]))
    assert list(bins_of(t1)) == [0, 10] and list(bins_of(t2)) == [0, 10] and list(bins_of(t3)) == [0, 10]
    edge = 2.0 * 3 / 11 - 1.0   # the edge between bins 2 and 3 of f2
    assert int(bins_of(11.0 * (edge + 1e-12 + 1.0) / 2.0)) == 3 and int(bins_of(11.0 * (edge - 1e-12 + 1.0) / 2.0)) == 2
    assert near_edge(11.0 * (edge + 1e-12 + 1.0) / 2.0)
    assert near_edge(np.array([3.0 + 1e-12, 3.5, 0.0, 11.0])).tolist() == [True, False, False, False]


def test_fpfh_restatement_on_a_hand_built_neighbourhood():
    # four points: a keypoint whose list holds a duplicate of itself (skipped in both sums) and a -1 (a cloud smaller than k)
    kp = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 0]], dtype=np.float32)
    nrm = np.array([[0, 0, 1], [0, 0.6, 0.8], [0.6, 0, 0.8], [0, 0, 1]], dtype=np.float32)
    nbr = np.array([[0, 3, 1, 2, -1], [1, 0, 3, 2, -1], [2, 0, 3, 1, -1], [0, 3, 1, 2, -1]], dtype=np.int64)
    f, edge = fpfh_numpy(kp, nrm, nbr, 5)
    assert not edge.any()
    # keypoint 0: its list gives 3, 1, 2 (itself excluded); the pair with the duplicate 3 has f4 == 0 and the duplicate's weight is
    # skipped, so each sub-histogram holds 2 pairs x 100 / 4 of its own and 100 of the weighted part; keypoint 1 has 3 pairs
    sums = np.stack([f[:, 11 * s:11 * s + 11].astype(np.float64).sum(1) for s in range(3)], axis=1)
    assert np.allclose(sums[0], 150.0) and np.allclose(sums[1], 175.0)
    assert np.array_equal(f[0], f[3])
    f2, _ = fpfh_numpy(kp, np.vstack([nrm[:3], [np.nan, 0, 0]]).astype(np.float32), nbr, 5)
    assert not f2[3].any() and f2[:3].any()


def test_pipeline_restatement_recovers_seeded_placements(synth):
    n = 20_000
    tgt = synth.full_object(n, seed=0x5EED0000 + 1, noise=0.2)
    obj = synth.full_object(n, seed=0x5EED0000 + 2, noise=0.2)
    for seed in range(4):
        P = synth.random_placement(seed)
        src = obj.copy()
        src[:, :3] = (obj[:, :3].astype(np.float64) @ P[:3, :3].T + P[:3, 3]).astype(np.float32)
        pose, matches = pipeline_numpy(src, tgt, seed)
        truth = np.linalg.inv(P)
        c = P[:3, :3] @ synth.CENTER + P[:3, 3]
        assert np.degrees(rot_angle(pose, truth)) < 5.0 and centre_error(pose, truth, c) < 5.0, (seed, matches)


def test_match_restatement_ties_and_zero_rows():
    a = np.zeros((3, 33), dtype=np.float32); a[0, 0] = 1; a[1, 5] = 2
    b = np.zeros((4, 33), dtype=np.float32); b[1, 0] = 1; b[2, 0] = 1; b[3, 5] = 2
    assert match_numpy(a, b).tolist() == [1, 3, -1]    # a tie goes to row 1; the zero query and the zero row never match
    assert match_numpy(a, b[:1]).tolist() == [-1, -1, -1]


def test_global_structs_match_the_header(mvr, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "mvr_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(mvr_global_params), '
                   'offsetof(mvr_global_params, max_dist), offsetof(mvr_global_params, hypotheses), offsetof(mvr_global_params, similarity), '
                   'offsetof(mvr_global_params, min_edge), offsetof(mvr_global_params, samples), offsetof(mvr_global_params, seed), '
                   'sizeof(mvr_global_report), offsetof(mvr_global_report, cost), offsetof(mvr_global_report, inliers), '
                   'offsetof(mvr_global_report, samples), offsetof(mvr_global_report, gpu_ms)); return 0; }\n')
    exe = str(tmp_path / "layout")
    r = subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    G, R = mvr.GlobalParams, mvr.GlobalReport
    assert got == [ctypes.sizeof(G), G.max_dist.offset, G.hypotheses.offset, G.similarity.offset, G.min_edge.offset, G.samples.offset,
                   G.seed.offset, ctypes.sizeof(R), R.cost.offset, R.inliers.offset, R.samples.offset, R.gpu_ms.offset]


def test_global_params_defaults(mvr):
    p = mvr.global_params()
    assert (p.keypoints, p.k, p.max_dist, p.hypotheses, p.max_draws, p.similarity, p.min_edge, p.samples) == \
        (4096, 32, 4.0, 2048, 1_000_000, 0.9, 0.05, 4096)
    assert mvr.global_params(seed=7, k=16).seed == 7


def test_synth_without_placement_is_unchanged(synth):
    views, poses = synth.turntable_sequence(5, 3000, placement=None)
    h = hashlib.sha256()
    for a in views:
        h.update(a.tobytes())
    for a in poses:
        h.update(np.ascontiguousarray(a).tobytes())
    assert h.hexdigest() == "756ba5991f2590ca99f99072fff08babefc79a1ef47d1dc2355b45b6a829cd60"
    P = synth.random_placement(5)
    assert np.allclose(P[:3, :3] @ P[:3, :3].T, np.eye(3)) and np.linalg.det(P[:3, :3]) > 0
    v, T = synth.turntable_view(2, 8, 2000, placement=P)
    assert np.allclose(T, np.linalg.inv(synth.rotation_about_axis(2 * 2 * np.pi / 8)))


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def _features(mvr, pts, which, keypoints, k, viewpoint=None):
    c = mvr.Context(0)
    (c.set_target if which == mvr.TARGET else c.set_source)(pts)
    out = c.fpfh(which, keypoints, k, viewpoint)
    c.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("k,keypoints", [(32, 4096), (8, 1000)])
def test_keypoint_normals_and_lists_equal_estimate_normals(mvr, synth, k, keypoints):
    pts, _ = synth.turntable_view(3, 24, 200_000)
    pts[17 * 49, :3] = np.nan   # a non-finite point at a keypoint slot: skipped
    c = mvr.Context(0)
    c.set_source(pts)
    idx, nrm, feat = c.fpfh(mvr.SOURCE, keypoints, k)
    assert np.array_equal(idx, keypoint_index(pts, keypoints))
    vp = (pts[np.isfinite(pts[:, :3]).all(1), :3].min(0) + pts[np.isfinite(pts[:, :3]).all(1), :3].max(0)) * np.float32(0.5)
    d = mvr.Context(0)
    d.set_target(pts[idx])
    want, nbr = d.estimate_normals(mvr.TARGET, len(idx), k, viewpoint=vp, want_neighbours=True)
    assert np.array_equal(nrm.view(np.uint32), want.view(np.uint32))
    # an explicit viewpoint at the box centre gives the same
    idx2, nrm2, feat2 = c.fpfh(mvr.SOURCE, keypoints, k, viewpoint=vp)
    assert np.array_equal(nrm2.view(np.uint32), nrm.view(np.uint32)) and np.array_equal(feat2.view(np.uint32), feat.view(np.uint32))
    want_f, edge = fpfh_numpy(pts[idx], nrm, nbr.astype(np.int64), k)
    take = taken_lists(nbr, k)
    shaky = edge.copy()
    shaky[np.nonzero((take & edge[np.where(nbr >= 0, nbr, 0)]).any(axis=1))[0]] = True
    assert edge.sum() <= 0.001 * len(idx), edge.sum()
    assert np.array_equal(feat[~shaky].view(np.uint32), want_f[~shaky].view(np.uint32))
    c.close(); d.close()


@pytest.mark.gpu
def test_match_features_equals_brute_force(mvr, synth):
    tgt, _ = synth.turntable_view(0, 8, 200_000)
    src, _ = synth.turntable_view(1, 8, 200_000)
    _, _, fa = _features(mvr, src, mvr.SOURCE, 4096, 32)
    _, _, fb = _features(mvr, tgt, mvr.TARGET, 3000, 16)
    fa, fb = fa.copy(), fb.copy()
    fb[10] = fb[20]; fb[30] = fb[20]                    # exact ties: the lowest row wins
    fa[5] = fb[20]
    fa[7] = 0; fb[40] = 0; fb[41] = fa[9]; fb[0] = 0    # all-zero rows on both sides
    c = mvr.Context(0)
    ab, ba = c.match_features(fa, fb)
    assert np.array_equal(ab, match_numpy(fa, fb)) and np.array_equal(ba, match_numpy(fb, fa))
    assert ab[5] == 10 and ab[7] == -1 and ab[9] == 41 and not (ab == 0).any() and ba[40] == -1
    e = np.zeros((0, 33), dtype=np.float32)
    ab, ba = c.match_features(fa[:100], e)
    assert (ab == -1).all() and len(ba) == 0
    c.close()


def _p2l_refine(mvr, c, tgt, src, pose, vp):
    c.estimate_normals(mvr.TARGET, len(tgt), 16, viewpoint=vp)
    p = mvr.default_params(max_iterations=60, max_dist=4.0, reciprocal=0, estimator=mvr.POINT_TO_PLANE, transformation_epsilon=1e-10)
    return c.icp_align(p, guess=pose, n_source=len(src))


def _place(pts, P):
    out = pts.copy()
    out[:, :3] = (pts[:, :3].astype(np.float64) @ P[:3, :3].T + P[:3, 3]).astype(np.float32)
    return out


@pytest.fixture(scope="module")
def full_clouds(synth):
    n = 200_000
    return synth.full_object(n, seed=0x5EED0000 + 1, noise=0.2), synth.full_object(n, seed=0x5EED0000 + 2, noise=0.2)


@pytest.fixture(scope="module")
def partial_views(synth):
    tgt, _ = synth.turntable_view(0, 8, 200_000)
    src, T1 = synth.turntable_view(1, 8, 200_000)
    return tgt, src, T1


def _check_recovery(mvr, tgt, src, truth, centre, vp):
    c = mvr.Context(0)
    c.set_target(tgt); c.set_source(src)
    pose, rep = c.global_align()
    assert rep["status"] == mvr.OK and rep["matches"] >= 3 and rep["hypotheses"] == 2048, rep
    ang, dc = np.degrees(rot_angle(pose, truth)), centre_error(pose, truth, centre)
    assert ang < 5.0 and dc < 5.0, (ang, dc, rep)
    r = _p2l_refine(mvr, c, tgt, src, pose, vp)
    assert rot_angle(r["final"], truth) < 2e-3 and centre_error(r["final"], truth, centre) < 1.0, (rot_angle(r["final"], truth), rep)
    c.close()
    return rep


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(8))
def test_global_align_recovers_full_object_placements(mvr, synth, full_clouds, seed):
    tgt, obj = full_clouds
    P = synth.random_placement(seed)
    _check_recovery(mvr, tgt, _place(obj, P), np.linalg.inv(P), P[:3, :3] @ synth.CENTER + P[:3, 3], synth.CENTER)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(8))
def test_global_align_recovers_partial_view_placements(mvr, synth, partial_views, seed):
    tgt, src0, T1 = partial_views
    P = synth.random_placement(100 + seed)
    _check_recovery(mvr, tgt, _place(src0, P), T1 @ np.linalg.inv(P), P[:3, :3] @ synth.CENTER + P[:3, 3], np.zeros(3))


@pytest.mark.gpu
def test_global_align_merges_two_rings_of_two_placements(mvr, synth):
    V, n = 12, 50_000
    reg = mvr.Registrator(0)
    icp = mvr.default_params(max_iterations=30, max_dist=4.0, reciprocal=1, fixed_iterations=1)
    prm = mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1)
    P = synth.random_placement(42)
    merged = []
    for placement in (None, P):
        views, _ = synth.turntable_sequence(V, n, placement=placement)
        poses, _ = reg.register_turntable(views, prm)
        c = mvr.Context(0)
        merged.append(np.concatenate([c.apply_pose(v, T.astype(np.float64)) for v, T in zip(views, poses)]))
        c.close()
    reg.close()
    _check_recovery(mvr, merged[0], merged[1], np.linalg.inv(P), P[:3, :3] @ synth.CENTER + P[:3, 3], synth.CENTER)


@pytest.mark.gpu
def test_global_align_same_bits_and_align_afterwards(mvr, synth, partial_views):
    tgt, src0, T1 = partial_views
    src = _place(src0, synth.random_placement(7))
    a, b = mvr.Context(0), mvr.Context(0)
    for c in (a, b):
        c.set_target(tgt); c.set_source(src)
    prm = mvr.global_params(hypotheses=700, seed=11)
    pa, ra = a.global_align(prm)
    pa2, ra2 = a.global_align(prm)
    pb, rb = b.global_align(prm)
    for r in (ra2, rb):
        assert {k: v for k, v in r.items() if k != "gpu_ms"} == {k: v for k, v in ra.items() if k != "gpu_ms"}
    assert np.array_equal(pa, pa2) and np.array_equal(pa, pb)
    assert ra["hypotheses"] == 700 and ra["samples"] > 0
    # the align after global_align: the same bits as on a fresh context
    f = mvr.Context(0)
    f.set_target(tgt); f.set_source(src)
    p = mvr.default_params(max_iterations=10, max_dist=4.0, reciprocal=1, fixed_iterations=1)
    x, y = a.icp_align(p, guess=pa, n_source=len(src)), f.icp_align(p, guess=pa, n_source=len(src))
    assert np.array_equal(x["final"], y["final"]) and x["n_corr"] == y["n_corr"] and x["mse"] == y["mse"]
    for c in (a, b, f):
        c.close()


@pytest.mark.gpu
def test_global_align_statuses(mvr, synth):
    pts, _ = synth.turntable_view(0, 8, 20_000)
    e = np.zeros((0, 4), dtype=np.float32)
    c = mvr.Context(0)
    with pytest.raises(mvr.MvrError) as ex:   # nothing set
        c.global_align()
    assert ex.value.status == mvr.ERR_NO_INPUT
    with pytest.raises(mvr.MvrError) as ex:
        c.fpfh(mvr.TARGET, 100, 16)
    assert ex.value.status == mvr.ERR_NO_INPUT
    c.set_target(pts)
    with pytest.raises(mvr.MvrError) as ex:   # no source
        c.global_align()
    assert ex.value.status == mvr.ERR_NO_INPUT
    c.set_source(e)                           # an empty source: no keypoints, no matches
    idx, nrm, feat = c.fpfh(mvr.SOURCE, 100, 16)
    assert len(idx) == 0 and feat.shape == (0, 33)
    pose, rep = c.global_align()
    assert rep["status"] == mvr.ERR_TOO_FEW and np.array_equal(pose, np.eye(4, dtype=np.float32)) and rep["matches"] == 0
    c.set_source(pts[:2])                     # two points: k_normals leaves their normals non-finite, nothing matches
    pose, rep = c.global_align(mvr.global_params(k=8))
    assert rep["status"] == mvr.ERR_TOO_FEW and np.array_equal(pose, np.eye(4, dtype=np.float32))
    c.set_source(pts)                         # no draw passes an impossible similarity
    pose, rep = c.global_align(mvr.global_params(keypoints=500, max_draws=200, similarity=1.0, min_edge=2.0))
    assert rep["status"] == mvr.ERR_TOO_FEW and rep["hypotheses"] == 0 and rep["draws"] == 200
    for bad in (dict(keypoints=0), dict(keypoints=65537), dict(k=7), dict(k=33), dict(samples=0), dict(similarity=1.5), dict(max_dist=0.0)):
        with pytest.raises(mvr.MvrError) as ex:
            c.global_align(mvr.global_params(**bad))
        assert ex.value.status == mvr.ERR_BAD_ARG
    c.close()
