"""Turntable ring registration from uncertain step angles: mvr_score_guesses_batch scores many candidate transforms of each
pair on the GPU (exact integer sums, compared for equality with a numpy restatement), and the ring driver's opt-in angle search
starts each pair from its best-scoring turn about the axis.  With the search off nothing changes."""
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MISS = 1 << 24
FLT_MAX = float(np.finfo(np.float32).max)


def rot_angle(A, B):
    R = np.asarray(A, dtype=np.float64)[:3, :3] @ np.asarray(B, dtype=np.float64)[:3, :3].T
    w = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return float(np.arcsin(min(1.0, np.linalg.norm(w))))


# ---- the cost, restated in numpy ---------------------------------------------------------------------------------------
def gate_float(max_dist):
    m2 = max_dist * max_dist
    if not m2 < FLT_MAX:
        return np.float32(np.inf)
    f = np.float32(m2)
    if float(f) < m2:
        f = np.nextafter(f, np.float32(np.inf))
    return np.nextafter(f, np.float32(np.inf))


def xform_pinned(M, p):
    """The align's float transform of points p (n x 3 float32) by the 4x4 M: ((m0 x + m1 y) + m2 z) + m3 per row, no FMA."""
    M = np.asarray(M, dtype=np.float32)
    x, y, z = p[:, 0], p[:, 1], p[:, 2]
    return np.stack([((M[r, 0] * x + M[r, 1] * y) + M[r, 2] * z) + M[r, 3] for r in range(3)], axis=1).astype(np.float32)


def d2_pinned(q, t):
    d = (q - t).astype(np.float32)
    return ((d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]).astype(np.float32)


def samples_of(src, samples):
    n = len(src)
    stride = max(1, -(-n // samples))
    p = np.asarray(src[::stride, :3], dtype=np.float32)
    return p[np.isfinite(p).all(axis=1)]


def sample_costs(min_d2, found, max_dist):
    """Per-sample cost from the exact float32 minimum distance (found: a target point exists)."""
    scale = np.float32(16777216.0 / float(gate_float(max_dist)))
    inl = found & ~(min_d2.astype(np.float64) > max_dist * max_dist)
    c = np.full(len(min_d2), MISS, dtype=np.uint64)
    c[inl] = np.minimum(np.floor(min_d2[inl].astype(np.float32) * scale).astype(np.uint64), MISS)
    return c, inl


def score_numpy(src, tgt, cands, max_dist, samples):
    """(costs, inliers) per candidate; candidates of the exact float32 minimum from scipy.spatial.cKDTree.query_ball_point."""
    from scipy.spatial import cKDTree
    if len(src) == 0 or len(tgt) == 0:
        return np.full(len(cands), samples << 24, dtype=np.uint64), np.zeros(len(cands), dtype=np.int64)
    p = samples_of(src, samples)
    t = np.asarray(tgt[:, :3], dtype=np.float32)
    t = t[np.isfinite(t).all(axis=1)]
    tree = cKDTree(t.astype(np.float64)) if len(t) else None
    costs, inls = [], []
    for M in cands:
        q = xform_pinned(M, p)
        fin = np.isfinite(q).all(axis=1)
        min_d2 = np.full(len(q), np.inf, dtype=np.float32)
        found = np.zeros(len(q), dtype=bool)
        if tree is not None and fin.any():
            qf = q[fin].astype(np.float64)
            dnn, _ = tree.query(qf, k=1)
            # every point whose pinned float distance can reach the float minimum lies within dnn (1 + 1e-5) in double
            near = dnn <= max_dist * (1.0 + 1e-5)
            md = np.full(int(fin.sum()), np.inf, dtype=np.float32)
            if near.any():
                balls = tree.query_ball_point(qf[near], dnn[near] * (1.0 + 1e-5) + 1e-9)   # each holds at least the double NN
                lens = np.array([len(b) for b in balls], dtype=np.int64)
                idx = np.concatenate([np.asarray(b, dtype=np.int64) for b in balls])
                d = d2_pinned(np.repeat(q[fin][near], lens, axis=0), t[idx])
                md[near] = np.minimum.reduceat(d, np.concatenate([[0], np.cumsum(lens)[:-1]]))
            min_d2[fin] = md
            found[fin] = near   # a point beyond the gate is never an inlier: "not found" costs the same
        c, inl = sample_costs(min_d2, found, max_dist)
        costs.append(int(c.sum()))
        inls.append(int(inl.sum()))
    return np.array(costs, dtype=np.uint64), np.array(inls, dtype=np.int64)


def score_brute(src, tgt, cands, max_dist, samples):
    """O(N M) reference: the pinned float32 distance to every target point."""
    if len(src) == 0 or len(tgt) == 0:
        return np.full(len(cands), samples << 24, dtype=np.uint64), np.zeros(len(cands), dtype=np.int64)
    p = samples_of(src, samples)
    t = np.asarray(tgt[:, :3], dtype=np.float32)
    t = t[np.isfinite(t).all(axis=1)]
    costs, inls = [], []
    for M in cands:
        q = xform_pinned(M, p)
        fin = np.isfinite(q).all(axis=1)
        if len(t):
            d = d2_pinned(q[:, None, :], t[None, :, :])
            md = np.where(fin, d.min(axis=1), np.float32(np.inf)).astype(np.float32)
            found = fin.copy()
        else:
            md = np.full(len(q), np.inf, dtype=np.float32)
            found = np.zeros(len(q), dtype=bool)
        c, inl = sample_costs(md, found, max_dist)
        costs.append(int(c.sum()))
        inls.append(int(inl.sum()))
    return np.array(costs, dtype=np.uint64), np.array(inls, dtype=np.int64)


def turn_candidates(synth, pose_t, pose_s, J, step):
    """H_j = inv(pose_t) R(j step) pose_s, j = -J..J, narrowed to float32 (the ring driver's candidates of a pair)."""
    inv = np.linalg.inv(pose_t)
    return np.stack([(inv @ synth.rotation_about_axis(j * step) @ pose_s).astype(np.float32) for j in range(-J, J + 1)])


# ---- CPU ---------------------------------------------------------------------------------------------------------------
def _small_case(seed=7):
    rng = np.random.default_rng(seed)
    tgt = np.ones((2000, 4), dtype=np.float32)
    tgt[:, :3] = rng.uniform(-20, 20, (2000, 3)).astype(np.float32)
    src = np.ones((1500, 4), dtype=np.float32)
    src[:, :3] = tgt[:1500, :3] + rng.normal(0, 1.0, (1500, 3)).astype(np.float32)
    # a sample exactly at the gate (d2 == 4 in float and double), one just beyond it, two equidistant target points (a tie),
    # non-finite points in both clouds
    tgt[0, :3] = (100, 100, 100); src[0, :3] = (102, 100, 100)
    tgt[1, :3] = (200, 100, 100); src[3, :3] = (np.nextafter(np.float32(202), np.float32(300)), 100, 100)
    tgt[2, :3] = (300, 101, 100); tgt[4, :3] = (300, 99, 100); src[6, :3] = (300, 100, 100)
    tgt[5, :3] = np.nan; tgt[6, 0] = np.inf
    src[9, :3] = np.nan; src[12, 1] = -np.inf
    return src, tgt


def _small_cands(rng_seed=3, nc=31):
    rng = np.random.default_rng(rng_seed)
    out = [np.eye(4, dtype=np.float32)]
    for a in range(1, nc):
        ang = rng.normal(0, 0.02, 3)
        th = np.linalg.norm(ang)
        k = ang / th
        K = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
        M = np.eye(4)
        M[:3, :3] = np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K
        M[:3, 3] = rng.normal(0, 1.0, 3)
        out.append(M.astype(np.float32))
    out.append(np.array([[1, 0, 0, np.inf], [0, 1, 0, 0], [0, 0, 1, 0], [0, 0, 0, 1]], dtype=np.float32))   # q not finite
    return np.stack(out)


@pytest.mark.parametrize("samples", [500, 4096])
def test_numpy_restatement_equals_brute_force(samples):
    src, tgt = _small_case()
    cands = _small_cands()
    a = score_numpy(src, tgt, cands, 2.0, samples)
    b = score_brute(src, tgt, cands, 2.0, samples)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    n_s = len(samples_of(src, samples))
    assert a[0][-1] == n_s * MISS and a[1][-1] == 0     # the non-finite candidate: every sample misses
    assert 0 < a[1][0] < n_s


def test_restated_cost_at_the_gate_and_the_empty_clouds():
    tgt = np.array([[0, 0, 0, 1], [10, 0, 0, 1], [10, 2, 0, 1], [10, -2, 0, 1]], dtype=np.float32)
    src = np.array([[2, 0, 0, 1], [np.nextafter(np.float32(2), np.float32(3)), 0, 0, 1], [10, 0, 0, 1], [np.nan, 0, 0, 1]], dtype=np.float32)
    I = np.eye(4, dtype=np.float32)[None]
    for f in (score_numpy, score_brute):
        c, i = f(src, tgt, I, 2.0, 4)
        scale = np.float32(16777216.0 / float(gate_float(2.0)))
        at_gate = int(np.floor(np.float32(4.0) * scale))
        assert at_gate < MISS
        assert int(c[0]) == at_gate + MISS + 0 and int(i[0]) == 2    # exactly at the gate: inside; just beyond: a miss; NaN: no sample
        assert f(src, tgt[:0], I, 2.0, 4)[0][0] == 4 << 24          # an empty target scores samples x 2^24
        assert f(src[:0], tgt, I, 2.0, 4)[0][0] == 4 << 24


def test_synth_without_angles_is_unchanged(synth):
    views, poses = synth.turntable_sequence(5, 3000)
    h = hashlib.sha256()
    for a in views:
        h.update(a.tobytes())
    for a in poses:
        h.update(np.ascontiguousarray(a).tobytes())
    assert h.hexdigest() == "756ba5991f2590ca99f99072fff08babefc79a1ef47d1dc2355b45b6a829cd60"
    v2, p2 = synth.turntable_sequence(5, 3000, angles=None)
    assert all(np.array_equal(a, b) for a, b in zip(views, v2))
    ang = synth.uneven_angles(5, 6.0)
    v3, p3 = synth.turntable_sequence(5, 3000, angles=ang)
    assert np.array_equal(v3[0], views[0])
    for v in range(5):
        assert np.allclose(p3[v], np.linalg.inv(synth.rotation_about_axis(ang[v])))


def test_angle_structs_match_the_header(mvr, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "mvr_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(mvr_angle_search), offsetof(mvr_angle_search, samples), '
                   'sizeof(mvr_angle_pick), offsetof(mvr_angle_pick, cost), offsetof(mvr_angle_pick, guess_cost), '
                   'offsetof(mvr_angle_pick, guess_inliers)); return 0; }\n')
    exe = str(tmp_path / "layout")
    r = subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [ctypes.sizeof(mvr.AngleSearch), mvr.AngleSearch.samples.offset, ctypes.sizeof(mvr.AnglePick), mvr.AnglePick.cost.offset,
                   mvr.AnglePick.guess_cost.offset, mvr.AnglePick.guess_inliers.offset]
    s = mvr.angle_search_default()
    assert abs(s.range - np.deg2rad(15)) < 1e-15 and abs(s.step - np.deg2rad(1)) < 1e-15 and s.samples == 4096


# ---- GPU: the scorer ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [50_000, 200_000])
def test_scorer_equals_the_numpy_restatement(mvr, synth, n):
    V = 24
    tgt, Tt = synth.turntable_view(0, V, n)
    src, Ts = synth.turntable_view(1, V, n)
    init_t, init_s = np.eye(4), synth.rotation_about_axis(-2 * np.pi / V)
    cands = turn_candidates(synth, init_t, init_s, 15, np.deg2rad(1.0))
    far = np.eye(4, dtype=np.float32); far[0, 3] = 1000.0
    cands[-1] = far                                      # no overlap at all
    c = mvr.Context(0)
    c.set_target(tgt); c.set_source(src)
    costs, inl, st = mvr.score_guesses_batch([c], cands[None], 4.0, 4096)
    assert st[0] == mvr.OK
    want_c, want_i = score_numpy(src, tgt, cands, 4.0, 4096)
    assert np.array_equal(costs[0], want_c) and np.array_equal(inl[0], want_i)
    n_s = len(samples_of(src, 4096))
    assert int(costs[0][-1]) == n_s * MISS and inl[0][-1] == 0
    assert int(np.argmin(costs[0][:-1])) in (14, 15, 16)   # the ideal turn scores best
    c.close()


@pytest.mark.gpu
def test_scorer_statuses_and_empty_clouds(mvr, synth):
    a, _ = synth.turntable_view(0, 24, 20_000)
    b, _ = synth.turntable_view(1, 24, 20_000)
    e = np.zeros((0, 4), dtype=np.float32)
    cs = [mvr.Context(0) for _ in range(4)]
    cs[0].set_target(a); cs[0].set_source(b)
    cs[1].set_target(e); cs[1].set_source(b)
    cs[2].set_target(a); cs[2].set_source(e)
    cs[3].set_target(a)                                   # no source
    cands = np.stack([np.eye(4, dtype=np.float32)] * 3)[None].repeat(4, axis=0)
    costs, inl, st = mvr.score_guesses_batch(cs, cands, 4.0, 1000)
    assert list(st) == [mvr.OK, mvr.OK, mvr.OK, mvr.ERR_NO_INPUT]
    assert all(int(x) == 1000 << 24 for x in costs[1]) and all(int(x) == 1000 << 24 for x in costs[2])
    assert not inl[1].any() and not inl[2].any()
    one, one_i, _ = mvr.score_guesses_batch([cs[0]], cands[:1], 4.0, 1000)
    assert np.array_equal(costs[0], one[0]) and np.array_equal(inl[0], one_i[0])
    for bad in (dict(samples=0), dict(samples=65537), dict(max_dist=-1.0)):
        kw = dict(max_dist=4.0, samples=1000); kw.update(bad)
        with pytest.raises(mvr.MvrError) as ex:
            mvr.score_guesses_batch([cs[0]], cands[:1], kw["max_dist"], kw["samples"])
        assert ex.value.status == mvr.ERR_BAD_ARG
    with pytest.raises(mvr.MvrError):
        mvr.score_guesses_batch([cs[0]], np.zeros((1, 1025, 4, 4), dtype=np.float32), 4.0, 1000)
    for c in cs:
        c.close()


@pytest.mark.gpu
def test_scorer_batch_of_60_equals_single_calls_and_builds_once(mvr, synth):
    V, n = 12, 8000
    views, poses = synth.turntable_sequence(V, n)
    cs = [mvr.Context(0) for _ in range(60)]
    cands = []
    for k, c in enumerate(cs):
        t, s = k % V, (k * 5 + 1) % V
        c.set_target(views[t]); c.set_source(views[s])
        cands.append(turn_candidates(synth, poses[t], poses[s], 3, np.deg2rad(2.0 + k % 3)))
    cands = np.stack(cands)
    before = mvr.kernel_launch_count()
    costs, inl, st = mvr.score_guesses_batch(cs, cands, 4.0, 2048)
    first = mvr.kernel_launch_count() - before
    assert (st == mvr.OK).all()
    before = mvr.kernel_launch_count()
    costs2, inl2, _ = mvr.score_guesses_batch(cs, cands, 4.0, 2048)
    assert mvr.kernel_launch_count() - before == 2           # unchanged targets: no index build, one score launch per 48 contexts
    assert first > 2
    assert np.array_equal(costs, costs2) and np.array_equal(inl, inl2)
    for k, c in enumerate(cs):
        one, one_i, _ = mvr.score_guesses_batch([c], cands[k:k + 1], 4.0, 2048)
        assert np.array_equal(one[0], costs[k]) and np.array_equal(one_i[0], inl[k]), k
    for c in cs:
        c.close()


@pytest.mark.gpu
def test_align_after_a_score_call_is_bit_identical(mvr, synth):
    n = 50_000
    tgt, _ = synth.turntable_view(0, 24, n)
    src, Ts = synth.turntable_view(1, 24, n)
    guess = (synth.perturbation() @ Ts).astype(np.float32)
    p = mvr.default_params(max_iterations=10, max_dist=4.0, reciprocal=1, fixed_iterations=1)
    a, b = mvr.Context(0), mvr.Context(0)
    for c in (a, b):
        c.set_target(tgt); c.set_source(src)
    mvr.score_guesses_batch([a], guess[None, None], 4.0, 4096)
    for c in (a, b):   # points the align's index builds take in (MVR_K_SORT units)
        c.set_profiling(True)
        c.kernel_stats(reset=True)
    ra = a.icp_align(p, guess=guess, n_source=n)
    rb = b.icp_align(p, guess=guess, n_source=n)
    built = [c.kernel_stats(reset=True)["sort"]["units"] for c in (a, b)]
    assert np.array_equal(ra["final"], rb["final"]) and ra["n_corr"] == rb["n_corr"] and ra["mse"] == rb["mse"]
    assert built == [n, 2 * n]                               # after the score call the align found its target index built
    a.close(); b.close()


# ---- GPU: the ring -----------------------------------------------------------------------------------------------------
# Per-view turn error of the uneven table, uniform in +-STEP_ERR_DEG (no other jitter on the guesses).  Point-to-plane's basin is
# wide: without the search it survives +-8 degrees on the bench workload and +-15 degrees with 50k points per view (DESIGN.md
# section 7).  The recovery test therefore runs the bench workload (24 x 200k) at +-15 degrees, pair step errors up to 25.3
# degrees, where one point-to-plane pair breaks without the search, and searches +-30 degrees; the invariance test keeps +-6.
STEP_ERR_DEG = 15.0
SEARCH_DEG = 30.0


def _tp(mvr, synth, est, **kw):
    icp = mvr.default_params(max_iterations=30, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=est)
    return mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1, **kw)


@pytest.fixture(scope="module")
def uneven(synth):
    V, n = 24, 200_000
    ang = synth.uneven_angles(V, STEP_ERR_DEG)
    views, poses = synth.turntable_sequence(V, n, angles=ang)
    return V, n, views, poses, synth.step_errors(V, STEP_ERR_DEG)


def _pair_errors(rep, poses, V):
    return np.array([rot_angle(rep[p]["pose"], np.linalg.inv(poses[p]) @ poses[(p + 1) % V]) for p in range(V)])


@pytest.mark.gpu
@pytest.mark.parametrize("est,med_tol,max_tol", [(1, 2e-4, 1e-3), (0, 2e-3, 5e-3)])
def test_ring_recovers_uneven_steps_with_the_search(mvr, synth, uneven, est, med_tol, max_tol):
    V, n, views, poses, err = uneven
    reg = mvr.Registrator(0, 1)
    _, rep_off = reg.register_turntable(views, _tp(mvr, synth, est))
    off = _pair_errors(rep_off, poses, V)
    assert reg.angle_search_log() == []
    assert off.max() > 1e-2, off.max()                       # without the search the ring does not survive these steps
    reg.set_angle_search(np.deg2rad(SEARCH_DEG), np.deg2rad(1.0), 4096)
    _, rep = reg.register_turntable(views, _tp(mvr, synth, est))
    on = _pair_errors(rep, poses, V)
    print("estimator %d: pair rotation error without the search median %.3g max %.3g, with it median %.3g max %.3g"
          % (est, np.median(off), off.max(), np.median(on), on.max()))
    assert all(r["status"] == mvr.OK for r in rep)
    assert np.median(on) <= med_tol and on.max() <= max_tol, (np.median(on), on.max())
    log = reg.angle_search_log()
    assert [r["pair"] for r in log] == list(range(V))
    step = np.deg2rad(1.0)
    for p, r in enumerate(log):
        true = err[p] - err[(p + 1) % V]
        assert abs(r["angle"] - true) <= step, (p, r["angle"], true)
        assert abs(r["angle"] - r["choice"] * step) < 1e-12 and r["cost"] <= r["guess_cost"]
        if r["choice"] == 0:
            assert r["cost"] == r["guess_cost"] and r["inliers"] == r["guess_inliers"]
    # the guess's record is the scorer's cost of the unchanged turntable guess
    cs = [mvr.Context(0) for _ in range(V)]
    for p, c in enumerate(cs):
        c.set_target(views[p]); c.set_source(views[(p + 1) % V])
    init = [np.eye(4)] + [mvr.turntable_rotation(synth.PIVOT, synth.AXIS, mvr.turntable_view_angle(v, V)) for v in range(1, V)]
    guess = np.stack([_driver_guess(init[p], init[(p + 1) % V])[None] for p in range(V)])
    costs, inl, st = mvr.score_guesses_batch(cs, guess, 4.0, 4096)
    for p, r in enumerate(log):
        assert int(costs[p, 0]) == r["guess_cost"] and int(inl[p, 0]) == r["guess_inliers"] and r["samples"] == len(samples_of(views[(p + 1) % V], 4096))
    for c in cs:
        c.close()
    reg.close()


def _driver_guess(init_t, init_s):
    """float(inverseRigid(pose_t) * pose_s) in the ring driver's arithmetic (double, its summation order)."""
    A = np.asarray(init_t, dtype=np.float64)
    inv = np.eye(4)
    inv[:3, :3] = A[:3, :3].T
    for i in range(3):
        inv[i, 3] = -((inv[i, 0] * A[0, 3] + inv[i, 1] * A[1, 3]) + inv[i, 2] * A[2, 3])
    B = np.asarray(init_s, dtype=np.float64)
    out = np.zeros((4, 4), dtype=np.float32)
    for r in range(4):
        for c in range(4):
            s = 0.0
            for k in range(4):
                s += inv[r, k] * B[k, c]
            out[r, c] = np.float32(s)
    return out


@pytest.mark.gpu
def test_search_off_and_never_set_give_the_same_bits(mvr, synth):
    V, n = 6, 8000
    views, poses = synth.turntable_sequence(V, n)
    tp = _tp(mvr, synth, mvr.POINT_TO_PLANE)
    a, b = mvr.Registrator(0, 1), mvr.Registrator(0, 1)
    pa, ra = a.register_turntable(views, tp)
    b.set_angle_search(np.deg2rad(10.0), np.deg2rad(1.0))
    b.set_angle_search(0.0)
    pb, rb = b.register_turntable(views, tp)
    assert b.angle_search_log() == []
    for p in range(V):
        assert np.array_equal(ra[p]["pose"], rb[p]["pose"]) and ra[p]["n_corr"] == rb[p]["n_corr"] and ra[p]["mse"] == rb[p]["mse"]
        assert np.array_equal(pa[p], pb[p])
    for bad in (dict(step=0.0), dict(step=-1.0), dict(step=np.deg2rad(0.01)), dict(samples=-1), dict(samples=70000)):
        kw = dict(range=np.deg2rad(10.0), step=np.deg2rad(1.0), samples=0); kw.update(bad)
        with pytest.raises(mvr.MvrError) as e:
            b.set_angle_search(kw["range"], kw["step"], kw["samples"])
        assert e.value.status == mvr.ERR_BAD_ARG
    a.close(); b.close()


@pytest.mark.gpu
def test_search_poses_do_not_depend_on_streams_grouping_ranges_or_gpus(mvr, synth):
    import torch
    import mvr_b200.ring as ring
    V, n = 8, 20_000
    views, poses = synth.turntable_sequence(V, n, angles=synth.uneven_angles(V, 6.0, seed=11))
    tp = _tp(mvr, synth, mvr.POINT_TO_PLANE)
    rng, step = np.deg2rad(15.0), np.deg2rad(1.0)
    reg1 = mvr.Registrator(0, 1)
    reg1.set_angle_search(rng, step)
    abs1, rep1 = reg1.register_turntable(views, tp)
    log1 = reg1.angle_search_log()
    assert len(log1) == V and any(r["choice"] != 0 for r in log1)
    reg4 = mvr.Registrator(0, 4)
    reg4.set_angle_search(rng, step)
    abs4, rep4 = reg4.register_turntable(views, tp)
    regg = mvr.Registrator(0, 1)
    regg.context(0).set_batch_group(1)
    regg.set_angle_search(rng, step)
    absg, repg = regg.register_turntable(views, tp)
    for reps, absv, log in ((rep4, abs4, reg4.angle_search_log()), (repg, absg, regg.angle_search_log())):
        assert log == log1
        for p in range(V):
            assert np.array_equal(reps[p]["pose"], rep1[p]["pose"]) and reps[p]["n_corr"] == rep1[p]["n_corr"] and reps[p]["mse"] == rep1[p]["mse"]
            assert np.array_equal(absv[p], abs1[p])
    got, glog = {}, []
    for lo, hi in ((0, 3), (3, 5), (5, 8)):
        need = {q % V for p in range(lo, hi) for q in (p, p + 1)}
        _, reps = reg4.register_turntable([views[v] if v in need else None for v in range(V)], _tp(mvr, synth, mvr.POINT_TO_PLANE, pair_begin=lo, pair_end=hi))
        glog += reg4.angle_search_log()
        for p in range(lo, hi):
            got[p] = reps[p]
    assert glog == log1
    for p in range(V):
        assert np.array_equal(got[p]["pose"], rep1[p]["pose"]) and got[p]["n_corr"] == rep1[p]["n_corr"]
    want = ring.pose_checksum(ring.pack_reports(rep1, 0, V))
    for g in [1] + [g for g in (2, 4, 8) if g <= torch.cuda.device_count()]:
        m = mvr.MultiRegistrator(range(g))
        m.set_angle_search(rng, step)
        got_poses, reps, recs, _ = m.register_turntable(views, tp)
        assert ring.pose_checksum(recs) == want, "%d GPUs: pair records differ from the single-GPU run" % g
        assert m.angle_search_log() == log1
        for a, b in zip(got_poses, abs1):
            assert np.array_equal(a, b)
        m.close()
    for r in (reg1, reg4, regg):
        r.close()
