"""CPU tests (no GPU): the C-ABI library loads and exports every symbol include/mvr_b200.h declares, fails loudly
without a CUDA device (no CPU fallback), and the pure host logic of the driver (turntable pose, ring closure, axis
refinement, sharding + gather over gloo) behaves as the reference's does."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_functions():
    txt = open(os.path.join(ROOT, "include", "mvr_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(mvr_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol(mvr):
    import ctypes
    L = mvr.lib()
    names = declared_functions()
    assert len(names) >= 40
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert b"sm_100a" in L.mvr_version()


def test_built_for_sm_100a_only():
    lib = os.path.join(ROOT, "multi-view-registration_b200", "libmvr_b200.so")
    out = subprocess.run(["cuobjdump", "-lelf", lib], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def _without_a_device(code):
    """Runs `code` in a child process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty), whether or not the machine has one."""
    r = subprocess.run([sys.executable, "-c", "import sys\nsys.path.insert(0, %r)\n%s" % (ROOT, code)],
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]


def test_no_cpu_fallback_without_a_device(mvr):
    _without_a_device(
        "import pytest\n"
        "import mvr_b200 as mvr\n"
        "with pytest.raises(mvr.MvrError):\n"
        "    mvr.Context(0)\n"
        "with pytest.raises(mvr.MvrError):\n"
        "    mvr.Registrator(0, 2)\n")


def test_product_never_touches_the_oracle():
    """The oracle is test infrastructure: nothing under the package or include/ may reference it."""
    bad = []
    for base in ("multi-view-registration_b200", "include"):
        for dp, _, fs in os.walk(os.path.join(ROOT, base)):
            for f in fs:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                    t = open(os.path.join(dp, f), errors="ignore").read()
                    if re.search(r"import oracle|from oracle|libmvr_oracle|orc_[a-z_]+\(", t):
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_turntable_rotation_and_view_angle(mvr):
    pivot, axis = [1.0, 2.0, 900.0], [0.0, -1.0, 0.0]
    for v in range(12):
        ref = ((-v) if v < 7 else (12 - v)) * np.pi / 6            # mvr/src/point_cloud.cpp:409
        assert mvr.turntable_view_angle(v, 12) == pytest.approx(ref, abs=1e-15)
    T = mvr.turntable_rotation(pivot, axis, 0.4)
    assert np.allclose(T @ np.array([1.0, 2.0, 900.0, 1.0]), [1.0, 2.0, 900.0, 1.0])      # the pivot is fixed
    assert np.allclose(T[:3, :3] @ np.array(axis), axis) and np.allclose(T[:3, :3].T @ T[:3, :3], np.eye(3))
    # right-handed rotation by +angle about the axis (osg::Matrix::rotate(angle, axis))
    e = np.array([1.0, 0.0, 0.0])
    assert np.allclose(np.cross(e, T[:3, :3] @ e) @ np.array(axis), np.sin(0.4))


def _ring(mvr, V, c):
    return [mvr.turntable_rotation(c, [0, -1, 0], -v * 2 * np.pi / V) for v in range(V)]


def test_ring_close_exact_chain_and_relaxation(mvr):
    rng = np.random.default_rng(1)
    V, c = 12, [0.0, 0.0, 900.0]
    X = _ring(mvr, V, c)
    rel = [np.linalg.inv(X[p]) @ X[(p + 1) % V] for p in range(V)]
    for relax in (False, True):
        out = mvr.ring_close(rel, relax=relax, centre=c, rot_scale=100.0)
        assert max(np.abs(out[v] - X[v]).max() for v in range(V)) < 5e-4      # float32 poses at |t| ~ 1800
    # one bad edge: chaining piles the whole error onto the views behind it, relaxation spreads it round the ring
    bad = [r.copy() for r in rel]
    bad[3] = bad[3] @ mvr.turntable_rotation(c, [0.1, 1.0, 0.2], 0.012)
    def ang(A, B):   # from the skew part: arccos of a float32 trace loses ~3e-4 rad
        R = np.asarray(A, float)[:3, :3] @ np.asarray(B, float)[:3, :3].T
        return float(np.arcsin(min(1.0, 0.5 * np.linalg.norm([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]]))))
    chain = mvr.ring_close(bad, relax=False)
    relaxed = mvr.ring_close(bad, relax=True, centre=c, rot_scale=100.0)
    assert max(ang(chain[v], X[v]) for v in range(V)) > 0.011
    assert max(ang(relaxed[v], X[v]) for v in range(V)) < 0.0085      # 0.012 * (V - 4) / V: the error is shared out
    # weights: a dropped edge (w = 0) takes all of the inconsistency, the rest is reproduced exactly
    w = [1.0] * V
    w[3] = 0.0
    dropped = mvr.ring_close(bad, w, relax=True, centre=c, rot_scale=100.0)
    assert max(ang(dropped[v], X[v]) for v in range(V)) < 1e-4


def test_refine_axis_recovers_the_turntable_axis(mvr):
    """Registrator::refineAxis (mvr/src/registrator.cpp:402-455) on exact turntable poses."""
    c, n = np.array([3.0, 7.0, 905.0]), np.array([0.05, 0.99, 0.1])
    n /= np.linalg.norm(n)
    poses = [mvr.turntable_rotation(c, n, mvr.turntable_view_angle(v, 12)) for v in range(1, 12)]
    pivot, axis = mvr.refine_axis(poses, pivot=[0.0, 7.0, 0.0], axis=[0.0, -1.0, 0.0])
    assert np.allclose(axis, n, atol=2e-6)              # u + v + w = 1 picks the sign with a positive sum
    # the pivot is only determined up to a slide along the axis; the reference pins its y to the old pivot's y
    assert pivot[1] == pytest.approx(7.0, abs=1e-4)
    d = pivot - c
    assert np.linalg.norm(d - (d @ n) * n) < 2e-3
    assert mvr.refine_axis([], [1, 2, 3], [0, -1, 0])[0].tolist() == [1, 2, 3]       # nothing registered: unchanged


def test_pack_unpack_records_and_pair_ranges(mvr):
    import mvr_b200.ring as ring
    for world in (1, 2, 3, 4, 8):
        seen = []
        for r in range(world):
            a, b = ring.pair_range(r, world, 24)
            seen += list(range(a, b))
        assert seen == list(range(24))
    assert ring.views_needed(22, 24, 24) == [0, 22, 23]
    reps = [dict(pose=np.eye(4) * (p + 1), n_corr=100 + p, mse=0.5 * p, iterations=30, status=0, nn_queries=(1 << 30) + p) for p in range(6)]
    back = ring.unpack_records(ring.pack_reports(reps, 2, 5))
    assert [b["n_corr"] for b in back] == [102, 103, 104] and back[0]["nn_queries"] == (1 << 30) + 2
    assert np.array_equal(back[1]["pose"], (np.eye(4) * 4).astype(np.float32))
    # the raw path (numpy view of the C report array, no per-pair Python objects) packs the same bytes, and the ring closes
    # the same from either
    raw = np.zeros(6, dtype=mvr.REPORT)
    rng = np.random.default_rng(3)
    for p in range(6):
        T = np.eye(4, dtype=np.float32); T[:3, 3] = rng.normal(size=3)
        reps[p]["pose"] = T
        raw[p]["pose"] = mvr.pose_from_numpy(T); raw[p]["n_correspondences"] = reps[p]["n_corr"]; raw[p]["mse"] = reps[p]["mse"]
        raw[p]["iterations"] = 30; raw[p]["status"] = 0; raw[p]["nn_queries"] = reps[p]["nn_queries"]
    a, b = ring.pack_reports(reps, 1, 6), ring.records_from_reports(raw, 1, 6)
    assert a.tobytes() == b.tobytes() and ring.pose_checksum(a) == ring.pose_checksum(b)
    flat = ring.close_ring(ring.pack_reports(reps, 0, 6), [0.0, 0.0, 0.0], 100.0)
    listed = mvr.ring_close([r["pose"] for r in reps], [float(r["n_corr"]) for r in reps], centre=[0.0, 0.0, 0.0], rot_scale=100.0)
    assert all(np.array_equal(x, y) for x, y in zip(flat, listed))


WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np, torch, torch.distributed as dist
import mvr_b200, mvr_b200.ring as ring
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=rank, world_size=world)
V, c = 10, [0.0, 0.0, 900.0]
rng = np.random.default_rng(7)          # same stream on every rank: the "measurements" of the whole ring
X = [mvr_b200.turntable_rotation(c, [0, -1, 0], -v * 2 * np.pi / V) for v in range(V)]
noise = [mvr_b200.turntable_rotation(c, rng.normal(size=3), 0.002 * rng.normal()) for _ in range(V)]
reps = [dict(pose=(np.linalg.inv(X[p]) @ X[(p + 1) % V] @ noise[p]).astype(np.float32), n_corr=1000 + p, mse=0.1, iterations=30, status=0,
             nn_queries=12345 + p) for p in range(V)]
p0, p1 = ring.pair_range(rank, world, V)
mine = ring.pack_reports(reps, p0, p1)          # every rank contributes ONLY its own block of pairs
allrec = ring.gather_records(mine, rank, world, V, dist=dist)
poses = ring.close_ring(allrec, c, 100.0)
np.save({out!r} + "_%d.npy" % rank, np.stack(poses))
dist.barrier()
dist.destroy_process_group()
"""


def test_sharded_ring_over_gloo_world_size_2_equals_single_process(tmp_path, mvr):
    """N > 1 path on CPU: pairs block-partitioned over 2 ranks, records all-gathered (gloo), ring closed on every rank."""
    import mvr_b200.ring as ring
    import socket
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = str(tmp_path / "poses")
    code = WORKER.format(root=ROOT, port=port, out=out)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        procs.append(subprocess.Popen([sys.executable, "-c", code], env=env))
    for p in procs:
        assert p.wait(timeout=180) == 0
    a, b = np.load(out + "_0.npy"), np.load(out + "_1.npy")
    assert np.array_equal(a, b)
    # single-process reference
    V, c = 10, [0.0, 0.0, 900.0]
    rng = np.random.default_rng(7)
    X = [mvr.turntable_rotation(c, [0, -1, 0], -v * 2 * np.pi / V) for v in range(V)]
    noise = [mvr.turntable_rotation(c, rng.normal(size=3), 0.002 * rng.normal()) for _ in range(V)]
    reps = [dict(pose=(np.linalg.inv(X[p]) @ X[(p + 1) % V] @ noise[p]).astype(np.float32), n_corr=1000 + p, mse=0.1, iterations=30, status=0,
                 nn_queries=12345 + p) for p in range(V)]
    one = ring.close_ring(ring.gather_records(ring.pack_reports(reps, 0, V), 0, 1, V), c, 100.0)
    assert np.array_equal(np.stack(one), a)


# ---- LUM relaxation on correspondence moments (lum.cpp lumRelax; reference mvr/src/registrator.cpp:627-663) ----------
def _rigid(rng, rot, trans):
    w = rot * rng.standard_normal(3)
    th = np.linalg.norm(w)
    K = np.array([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
    R = np.eye(3) + np.sin(th) / th * K + (1 - np.cos(th)) / th ** 2 * (K @ K)
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = trans * rng.standard_normal(3)
    return T


def _apply(T, p):
    return p @ T[:3, :3].T + T[:3, 3]


def test_pair_moments_transform_matches_moments_of_transformed_pairs(mvr):
    rng = np.random.default_rng(3)
    a = rng.standard_normal((500, 3)) * 40 + [0, 0, 900]
    b = a + rng.standard_normal((500, 3))
    T = _rigid(rng, 0.7, 50.0)
    m = mvr.PairMoments.from_pairs(a, b, origin=[1, 2, 880])
    got = mvr.pair_moments_transform(m, T, new_origin=[5, -3, 20]).as_dict()
    want = mvr.PairMoments.from_pairs(_apply(T, a), _apply(T, b), origin=[5, -3, 20]).as_dict()
    for k in ("n", "sa", "sb", "sba", "saa", "sbb", "d2"):
        np.testing.assert_allclose(got[k], want[k], rtol=1e-10, atol=1e-6)
    keep = mvr.pair_moments_transform(m, T).as_dict()   # default origin: pose * old origin
    np.testing.assert_allclose(keep["origin"], _apply(T, np.array([[1.0, 2.0, 880.0]]))[0], atol=1e-9)


def test_lum_relax_recovers_known_corrections_from_exact_pairs(mvr):
    """Same surface points seen by both ends of every ring edge, views displaced rigidly: the relaxation must undo it."""
    rng = np.random.default_rng(11)
    V = 5
    truth = [np.eye(4)] + [_rigid(rng, 0.01, 0.8) for _ in range(V - 1)]   # displacement D_v of view v (world frame)
    edges, src, tgt = [], [], []
    for i in range(V):
        s, t = i, (i + 1) % V
        p = rng.standard_normal((300, 3)) * 60 + [0, 0, 900]
        edges.append(mvr.PairMoments.from_pairs(_apply(truth[s], p), _apply(truth[t], p), origin=[0, 0, 900]))
        src.append(s); tgt.append(t)
    X = mvr.lum_relax(edges, src, tgt, V, 16)
    np.testing.assert_allclose(X[0], np.eye(4), atol=0)
    for v in range(1, V):
        np.testing.assert_allclose(X[v] @ truth[v], np.eye(4), atol=1e-8)   # X_v = D_v^-1 (D_0 = I fixes the gauge)


def test_lum_relax_minimises_the_pair_cost_like_a_generic_solver(mvr):
    from scipy.optimize import least_squares
    from scipy.spatial.transform import Rotation
    rng = np.random.default_rng(5)
    V = 4
    disp = [np.eye(4)] + [_rigid(rng, 0.02, 1.0) for _ in range(V - 1)]
    pairs, edges, src, tgt = [], [], [], []
    for (s, t) in [(0, 1), (1, 2), (2, 3), (3, 0), (0, 2)]:          # a ring plus a chord: any graph is allowed
        p = rng.standard_normal((200, 3)) * 50 + [0, 0, 900]
        a = _apply(disp[s], p) + 0.3 * rng.standard_normal(p.shape)   # noisy: the optimum has a non-zero residual
        b = _apply(disp[t], p) + 0.3 * rng.standard_normal(p.shape)
        pairs.append((s, t, a, b))
        edges.append(mvr.PairMoments.from_pairs(a, b, origin=[0, 0, 900]))
        src.append(s); tgt.append(t)

    def pose(x6):
        T = np.eye(4)
        T[:3, :3] = Rotation.from_rotvec(x6[:3]).as_matrix()
        T[:3, 3] = x6[3:]
        return T

    def resid(x):
        Xs = [np.eye(4)] + [pose(x[6 * k:6 * k + 6]) for k in range(V - 1)]
        return np.concatenate([(_apply(Xs[s], a) - _apply(Xs[t], b)).ravel() for (s, t, a, b) in pairs])

    sol = least_squares(resid, np.zeros(6 * (V - 1)), xtol=1e-14, ftol=1e-14, gtol=1e-14)
    X = mvr.lum_relax(edges, src, tgt, V, 16)
    cost = lambda Xs: sum(((_apply(Xs[s], a) - _apply(Xs[t], b)) ** 2).sum() for (s, t, a, b) in pairs)
    c_lum, c_ref, c_0 = cost(X), 2.0 * sol.cost, cost([np.eye(4)] * V)
    assert c_lum < 0.5 * c_0 and abs(c_lum - c_ref) <= 1e-9 * c_ref
    for v in range(1, V):
        np.testing.assert_allclose(X[v], pose(sol.x[6 * (v - 1):6 * v]), atol=1e-6)


def test_lum_relax_edge_cases(mvr):
    X = mvr.lum_relax([], [], [], 3, 16)                       # no edges: nothing moves
    assert all(np.array_equal(x, np.eye(4)) for x in X)
    empty = mvr.PairMoments()                                  # an edge without correspondences carries no information
    rng = np.random.default_rng(2)
    p = rng.standard_normal((50, 3)) * 30
    D = _rigid(rng, 0.01, 0.5)
    e01 = mvr.PairMoments.from_pairs(p, _apply(D, p))
    X = mvr.lum_relax([e01, empty], [0, 1], [1, 2], 3, 16)
    np.testing.assert_allclose(X[1] @ D, np.eye(4), atol=1e-8)  # view 1 follows its only edge
    np.testing.assert_allclose(X[2], np.eye(4), atol=1e-12)     # view 2 is unconstrained: stays
    with pytest.raises(mvr.MvrError):
        mvr.lum_relax([e01], [0], [3], 3, 16)                   # view index out of range


def test_lum_outer_loops_descend_steadily_on_oracle_correspondences(mvr, orc, synth):
    """registrationLUM's loop (reciprocal correspondences -> moments -> 16 sweeps -> pose update), with the oracle's
    correspondences: the mean pair distance and the pose error fall loop after loop (the former pose-graph
    approximation of the edges diverged here after five loops)."""
    V, n = 6, 4000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    P = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]

    def rot_err(Pv):
        out = []
        for v in range(V):
            R = (np.linalg.inv(Pv[0]) @ Pv[v])[:3, :3] @ (np.linalg.inv(poses[0]) @ poses[v])[:3, :3].T
            out.append(np.arcsin(min(1.0, 0.5 * np.linalg.norm([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]]))))
        return max(out)

    e0, msd = rot_err(P), []
    for loop in range(10):
        edges = []
        for i in range(V):
            s, t = i, (i + 1) % V
            guess = (np.linalg.inv(P[t]) @ P[s]).astype(np.float32)
            a = orc.transform(views[s], guess)
            q, m, _ = orc.correspondences(a, views[t], 6.0, True)
            mom = mvr.PairMoments.from_pairs(a[q, :3], views[t][m, :3], origin=synth.PIVOT)
            edges.append(mvr.pair_moments_transform(mom, P[t]))
        msd.append(sum(e.d2 for e in edges) / sum(e.n for e in edges))
        X = mvr.lum_relax(edges, list(range(V)), [(i + 1) % V for i in range(V)], V, 16)
        P = [X[v] @ P[v] for v in range(V)]
    assert e0 > 0.02 and rot_err(P) < 0.75 * e0
    assert all(b < a * 1.01 for a, b in zip(msd, msd[1:])) and msd[-1] < 0.7 * msd[0]


# ---- persistence in the reference's text formats (mvr/src/point_cloud.cpp:305-347, mvr/src/registrator.cpp:258-328, 385-395) ----
def test_transformation_txt_format_and_round_trip(mvr, tmp_path):
    T = np.array([[0.5, -0.8660254, 0.0, 12.25], [0.8660254, 0.5, 0.0, -3.5], [0.0, 0.0, 1.0, 900.125], [0.0, 0.0, 0.0, 1.0]])
    f = tmp_path / "transformation.txt"
    mvr.transformation_save(f, T)
    # the reference prints matrix(j, i) of its row-vector matrix with "%lf ": the column-vector matrix row by row
    want = "".join("".join("%f " % T[i, j] for j in range(4)) + "\n" for i in range(4))
    assert f.read_text() == want
    np.testing.assert_allclose(mvr.transformation_load(f), T, atol=5e-7)
    # a file the reference wrote (hand-made here): element (i, j) is the j-th number of line i
    g = tmp_path / "ref.txt"
    g.write_text("1 0 0 5\n0 0 -1 6\n0 1 0 7\n0 0 0 1\n")
    np.testing.assert_array_equal(mvr.transformation_load(g), [[1, 0, 0, 5], [0, 0, -1, 6], [0, 1, 0, 7], [0, 0, 0, 1]])
    with pytest.raises(mvr.MvrError):
        mvr.transformation_load(tmp_path / "missing.txt")
    (tmp_path / "short.txt").write_text("1 2 3\n")
    with pytest.raises(mvr.MvrError):
        mvr.transformation_load(tmp_path / "short.txt")


def test_axis_txt_format_and_round_trip(mvr, tmp_path):
    f = tmp_path / "axis.txt"
    mvr.axis_save(f, [-13.382786, 50.223461, 917.4776], [-0.054323, -0.814921, -0.57702])
    assert f.read_text() == "-13.382786 50.223461 917.477600\n-0.054323 -0.814921 -0.577020\n"
    pv, ax = mvr.axis_load(f)
    np.testing.assert_allclose(pv, [-13.382786, 50.223461, 917.4776], atol=1e-6)
    np.testing.assert_allclose(ax, [-0.054323, -0.814921, -0.57702], atol=1e-6)


def test_points_asc_format(mvr, tmp_path):
    pts = np.zeros(2, dtype=mvr.RICH_POINT)
    pts["x"], pts["y"], pts["z"] = [1.5, -2.25], [0.0, 3.0], [900.0, 901.5]
    pts["r"], pts["g"], pts["b"] = [255, 1], [128, 2], [0, 3]
    f = tmp_path / "points.asc"
    mvr.points_save_asc(f, pts)
    assert f.read_text() == "1.500000 0.000000 900.000000 255 128 0\n-2.250000 3.000000 901.500000 1 2 3\n"


def test_lum_relax_golden(mvr):
    """tests/golden/lum.npz: explicit point pairs of a 5-view graph and the minimiser scipy.optimize.least_squares found
    (tests/golden/make_golden.py lum_fixture); the library sees the pairs only through their moments."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "lum.npz"))
    edges = [mvr.PairMoments.from_pairs(a, b, origin=[0, 0, 900]) for a, b in zip(g["a"], g["b"])]
    X = mvr.lum_relax(edges, g["src"], g["tgt"], len(g["X"]), 16)
    for v in range(len(g["X"])):
        np.testing.assert_allclose(X[v], g["X"][v], atol=2e-6)   # the accuracy scipy stopped at
    cost = sum((((a @ X[s][:3, :3].T + X[s][:3, 3]) - (b @ X[t][:3, :3].T + X[t][:3, 3])) ** 2).sum()
               for s, t, a, b in zip(g["src"], g["tgt"], g["a"], g["b"]))
    assert abs(cost - float(g["cost"])) <= 1e-9 * float(g["cost"])


def test_pair_record_layout_matches_the_header(mvr):
    """mvr_pair_record is exchanged as raw bytes: the ctypes mirror, the numpy dtype of ring.py and the C struct are all 96 bytes
    with the same field offsets."""
    import ctypes
    import mvr_b200.ring as ring
    assert ctypes.sizeof(mvr.PairRecord) == ring.REC == 96
    for name, np_name in (("pose", "pose"), ("n_correspondences", "n_corr"), ("iterations", "iterations"), ("status", "status"),
                          ("mse", "mse"), ("nn_queries", "nn_queries")):
        assert getattr(mvr.PairRecord, name).offset == ring.RECORD.fields[np_name][1]
    for rank, world, n in ((0, 1, 24), (3, 8, 24), (7, 8, 24), (1, 5, 7)):
        a, b = ctypes.c_int(0), ctypes.c_int(0)
        mvr.lib().mvr_multi_pair_range(rank, world, n, ctypes.byref(a), ctypes.byref(b))
        assert (a.value, b.value) == ring.pair_range(rank, world, n)


def test_multi_create_without_gpu_fails_loudly(mvr):
    _without_a_device(
        "import ctypes\n"
        "import mvr_b200 as mvr\n"
        "h = ctypes.c_void_p()\n"
        "assert mvr.lib().mvr_multi_create(None, 2, ctypes.byref(h)) == mvr.ERR_CUDA and not h.value\n")


def _lum_ring(orc, synth, V=6, n=6000):
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    clouds = [orc.apply_pose_double(views[v], init[v]) for v in range(V)]
    edges = []
    for i in range(V):
        s, t = i, (i + 1) % V
        iq, im, _ = orc.correspondences(clouds[s], clouds[t], 4.0, True)
        edges.append((s, t, iq, im))
    return views, poses, init, clouds, edges


def test_lum_oracle_edge_model_is_the_exact_linearisation(orc):
    """The restated computeEdge / incidenceCorrection pair (oracle/lum_oracle.py) is Borrmann et al.'s linearisation: for
    R = Rx Ry Rz the Jacobian of a compounded point with respect to (x, y, z, roll, pitch, yaw) equals M(point) * H(pose)."""
    import lum_oracle as L
    rng = np.random.default_rng(0)
    for _ in range(5):
        p = np.concatenate([rng.normal(size=3) * 5, rng.normal(size=3) * 0.4])
        x = rng.normal(size=3) * 50

        def f(q):
            ca, sa, cb, sb, cc, sc = np.cos(q[3]), np.sin(q[3]), np.cos(q[4]), np.sin(q[4]), np.cos(q[5]), np.sin(q[5])
            Rx = np.array([[1, 0, 0], [0, ca, -sa], [0, sa, ca]]); Ry = np.array([[cb, 0, sb], [0, 1, 0], [-sb, 0, cb]])
            Rz = np.array([[cc, -sc, 0], [sc, cc, 0], [0, 0, 1]])
            return Rx @ Ry @ Rz @ x + q[:3]
        J = np.stack([(f(p + 1e-6 * e) - f(p - 1e-6 * e)) / 2e-6 for e in np.eye(6)], axis=1)
        a = f(p)
        M = np.array([[1, 0, 0, 0, -a[1], a[2]], [0, 1, 0, -a[2], a[0], 0], [0, 0, 1, a[1], 0, -a[0]]])
        assert np.abs(J - M @ L.incidence_correction(p)).max() < 1e-6 * np.abs(J).max()
    # pcl::getTransformation is Translation * Rz(yaw) * Ry(pitch) * Rx(roll)
    T = L.get_transformation([1, 2, 3, 0.1, 0.2, 0.3])
    from scipy.spatial.transform import Rotation
    assert np.allclose(T[:3, :3], Rotation.from_euler("ZYX", [0.3, 0.2, 0.1]).as_matrix()) and np.allclose(T[:3, 3], [1, 2, 3])


def test_lum_compute_on_moments_equals_the_point_level_oracle(mvr, orc, synth):
    """mvr_lum_compute (pcl::registration::LUM's sweeps on 30 doubles per edge) against oracle/lum_oracle.py, which walks the
    correspondence lists like PCL's computeEdge: poses after 1, 5 and 16 sweeps agree to rounding; and the sweeps close the
    ring (the drift of the perturbed poses shrinks)."""
    import lum_oracle as L
    views, poses, init, clouds, edges = _lum_ring(orc, synth)
    V = len(views)
    mom = [mvr.PairMoments.from_pairs(clouds[s][iq, :3], clouds[t][im, :3], origin=clouds[t][:, :3].mean(axis=0).astype(np.float64))
           for (s, t, iq, im) in edges]
    for sweeps in (1, 5, 16):
        p6, X = mvr.lum_compute(mom, [e[0] for e in edges], [e[1] for e in edges], V, sweeps)
        o6, OX = L.lum_compute(clouds, edges, max_iterations=sweeps)
        # absolute coordinates of ~900 mm make M'M ill-conditioned: rounding level here is ~1e-8 mm / ~1e-11 rad
        assert np.abs(p6[:, :3] - o6[:, :3]).max() < 1e-6 and np.abs(p6[:, 3:] - o6[:, 3:]).max() < 1e-9
        for a, b in zip(X, OX):
            assert np.abs(a - b).max() < 1e-6
    assert np.all(p6[0] == 0)   # vertex 0 is the reference
    # one edge without correspondences, one view without edges: no information, the rest still solves
    mom2 = list(mom); mom2[2] = mvr.PairMoments()
    p6b, _ = mvr.lum_compute(mom2, [e[0] for e in edges], [e[1] for e in edges], V, 4)
    o6b, _ = L.lum_compute(clouds, [e if k != 2 else (e[0], e[1], e[2][:0], e[3][:0]) for k, e in enumerate(edges)], max_iterations=4)
    assert np.abs(p6b[:, :3] - o6b[:, :3]).max() < 1e-6 and np.abs(p6b[:, 3:] - o6b[:, 3:]).max() < 1e-9


def test_registration_lum_oracle_loop_reduces_drift(orc, synth):
    """The reference's registrationLUM loop restated on the CPU (oracle/lum_oracle.registration_lum): the ring error against the
    true poses falls with the number of outer loops."""
    import lum_oracle as L
    views, poses, init, _, _ = _lum_ring(orc, synth, n=6000)
    V = len(views)

    def err(P):
        out = 0.0
        for v in range(V):
            R = (np.linalg.inv(P[0]) @ P[v])[:3, :3] @ (np.linalg.inv(poses[0]) @ poses[v])[:3, :3].T
            w = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
            out = max(out, float(np.arcsin(min(1.0, np.linalg.norm(w)))))
        return out
    e0 = err(init)
    e4 = err(L.registration_lum(views, init, 64, 4.0, orc.correspondences, orc.apply_pose_double))
    e10 = err(L.registration_lum(views, init, 160, 4.0, orc.correspondences, orc.apply_pose_double))
    assert e10 < e4 < e0 and e10 < 0.75 * e0


def _build_adapter_check(tmp_path):
    import subprocess
    exe = str(tmp_path / "adapter_check")
    libdir = os.path.join(ROOT, "multi-view-registration_b200")
    cmd = ["g++", "-std=c++11", "-I" + os.path.join(ROOT, "include"), "-I" + os.path.join(ROOT, "tests", "mock_pcl"),
           os.path.join(ROOT, "tests", "adapter_check.cpp"), "-o", exe, os.path.join(libdir, "libmvr_b200.so"), "-Wl,-rpath," + libdir]
    for d in ("/usr/local/cuda/lib64", "/usr/local/cuda/targets/x86_64-linux/lib"):
        if os.path.isdir(d):
            cmd += ["-L" + d, "-Wl,-rpath," + d]
    r = subprocess.run(cmd + ["-lcudart"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return exe


def test_pcl_adapter_header_compiles_and_links(mvr, tmp_path):
    """include/mvr_pcl_adapter.hpp (the GpuICP / GpuCorrespondenceEstimation classes a maintainer puts under
    mvr/include/registrator.h:91 and mvr/src/registrator.cpp:496, 551, 644) is real C++: compiled against stand-in PCL / Eigen
    declarations and linked with the library; without a GPU its constructor fails loudly."""
    import subprocess
    import torch
    mvr.lib()
    exe = _build_adapter_check(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0, out.stderr
    if not torch.cuda.is_available():
        assert "no usable CUDA device" in out.stdout


def test_bench_reference_arm_prints_the_contract_line():
    """bench.py --impl reference (the CPU oracle port timed on the host cores) on a tiny configuration: one JSON line with the
    keys the driver reads; under torchrun only rank 0 prints."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--views", "4", "--points", "3000", "--iters", "4",
           "--steps", "1", "--warmup", "0", "--cpu-sample-pairs", "2"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=dict(os.environ, RANK="0"))
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "queries/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["views"] == 4 and d["config"]["points_per_view"] == 3000
    quiet = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=dict(os.environ, RANK="1"))
    assert quiet.returncode == 0 and quiet.stdout.strip() == ""
