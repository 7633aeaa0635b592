"""Symmetric point-to-plane ICP (MVR_SYMMETRIC): PCL's TransformationEstimationSymmetricPointToPlaneLLS with
enforce_same_direction_normals, the source normals moving with the source.  CPU: the oracle's step, pose construction and loop
against numpy / scipy restatements.  GPU: single aligns and batches against the oracle given the GPU's own normals, the three
ways of giving source normals, the missing-normals errors, and the ring driver (hand-built pairs, streams, grouping, shards,
GPU count, accuracy at bench size)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.spatial import cKDTree
from scipy.spatial.transform import Rotation

ROT_TOL = 1e-5       # rad
TRANS_REL_TOL = 1e-6


def rot_angle(A, B):
    R = np.asarray(A, dtype=np.float64)[:3, :3] @ np.asarray(B, dtype=np.float64)[:3, :3].T
    w = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return float(np.arcsin(min(1.0, np.linalg.norm(w))))


def driver_guess(init_t, init_s):
    """The ring driver's initial guess of a pair in its arithmetic (see test_point_to_plane_ring.py)."""
    A = [[float(init_t[r, c]) for c in range(4)] for r in range(4)]
    B = [[float(init_s[r, c]) for c in range(4)] for r in range(4)]
    inv = [[1.0 if r == c else 0.0 for c in range(4)] for r in range(4)]
    for i in range(3):
        for j in range(3):
            inv[i][j] = A[j][i]
    for i in range(3):
        inv[i][3] = -((inv[i][0] * A[0][3] + inv[i][1] * A[1][3]) + inv[i][2] * A[2][3])
    out = np.zeros((4, 4), dtype=np.float32)
    for r in range(4):
        for c in range(4):
            s = 0.0
            for k in range(4):
                s += inv[r][k] * B[k][c]
            out[r, c] = np.float32(s)
    return out


# ---- the CPU checker of the symmetric estimator: tests/symmetric_oracle.cpp (the oracle plus the symmetric step and loop) ----
HERE = os.path.dirname(os.path.abspath(__file__))


class SymOracle:
    """ctypes binding of tests/symmetric_oracle.cpp, built into a temporary directory."""

    def __init__(self, orc, path):
        self.orc = orc   # oracle/oracle.py: IcpParams, IcpReport, IterRecord, make_params
        L = C.CDLL(path)
        fp, dp, ip = C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.sym_estimate.argtypes = [fp, fp, fp, fp, ip, ip, C.c_int, dp, dp]
        L.sym_estimate.restype = C.c_int
        L.sym_icp_align.argtypes = [fp, fp, C.c_int, fp, C.c_int, fp, C.POINTER(orc.IcpParams), fp, fp, C.POINTER(orc.IcpReport),
                                    C.POINTER(orc.IterRecord), C.c_int, ip]
        L.sym_icp_align.restype = C.c_int
        self.lib = L

    @staticmethod
    def _pts(a):
        a = np.ascontiguousarray(a, dtype=np.float32)
        assert a.ndim == 2 and a.shape[1] == 4
        return a

    @staticmethod
    def _f(a):
        return a.ctypes.data_as(C.POINTER(C.c_float))

    def estimate_symmetric(self, src, src_normals, tgt, tgt_normals, q, m):
        """One step over the correspondences (q[k] source, m[k] target): (rc, T 4x4, x 6); rc 1 = not positive definite."""
        src, sn, tgt, tn = (self._pts(a) for a in (src, src_normals, tgt, tgt_normals))
        q = np.ascontiguousarray(q, dtype=np.int32)
        m = np.ascontiguousarray(m, dtype=np.int32)
        T = np.empty(16); x = np.zeros(6)
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
        rc = self.lib.sym_estimate(self._f(src), self._f(sn), self._f(tgt), self._f(tn), q.ctypes.data_as(ip), m.ctypes.data_as(ip), len(q),
                                   T.ctypes.data_as(dp), x.ctypes.data_as(dp))
        return rc, T.reshape(4, 4).T.copy(), x

    def icp_align(self, src, src_normals, tgt, tgt_normals, params, guess=None, max_log=256):
        """The oracle's ICP loop with the symmetric estimator; returns a dict like oracle.icp_align."""
        src, sn, tgt, tn = (self._pts(a) for a in (src, src_normals, tgt, tgt_normals))
        assert len(sn) == len(src) and len(tn) == len(tgt)
        g = np.eye(4, dtype=np.float32) if guess is None else np.asarray(guess, dtype=np.float32)
        gc = np.ascontiguousarray(g.T)
        fin = np.empty(16, dtype=np.float32)
        rep = self.orc.IcpReport()
        log = (self.orc.IterRecord * max_log)()
        nlog = C.c_int(0)
        rc = self.lib.sym_icp_align(self._f(src), self._f(sn), len(src), self._f(tgt), len(tgt), self._f(tn), C.byref(params), self._f(gc),
                                    self._f(fin), C.byref(rep), log, max_log, C.byref(nlog))
        recs = [dict(iteration=log[k].iteration, n_corr=log[k].n_corr, mse=log[k].mse,
                     delta=np.array(log[k].delta[:], dtype=np.float64).reshape(4, 4).T.copy()) for k in range(nlog.value)]
        return dict(status=rc, final=fin.reshape(4, 4).T.copy(), iterations=rep.iterations, reason=rep.reason,
                    n_corr=rep.n_correspondences, mse=rep.mse, log=recs)


@pytest.fixture(scope="module")
def sym(orc, tmp_path_factory):
    out = str(tmp_path_factory.mktemp("symmetric_oracle") / "libsymmetric_oracle.so")
    base = ["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-o", out,
            os.path.join(HERE, "symmetric_oracle.cpp")]
    r = subprocess.run(base[:1] + ["-fopenmp"] + base[1:], capture_output=True, text=True)
    if r.returncode != 0:   # no OpenMP: the same arithmetic, one thread (as oracle/Makefile does)
        r = subprocess.run(base, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return SymOracle(orc, out)


# ---- numpy restatement --------------------------------------------------------------------------------------------------
def rzyx(x):
    """R = Rz(x2) Ry(x1) Rx(x0), the rotation of pose_from_6."""
    return Rotation.from_euler("ZYX", [x[2], x[1], x[0]]).as_matrix()


def np_symmetric_step(p, n1, q, n2):
    """One step: p, q, n1, n2 are k x 3 float64.  Returns (T 4x4, x)."""
    same = np.sum(n1 * n2, axis=1) >= 0
    n = np.where(same[:, None], n1 + n2, n1 - n2)
    ok = np.all(np.isfinite(n), axis=1)
    p, q, n = p[ok], q[ok], n[ok]
    v = np.hstack([np.cross(p + q, n), n])
    r = np.sum((q - p) * n, axis=1)
    x = np.linalg.solve(v.T @ v, v.T @ r)
    R = rzyx(x)
    T = np.eye(4)
    T[:3, :3] = R @ R
    T[:3, 3] = R @ x[3:]
    return T, x


def xform_f32(M, p):
    """The pinned float transform: ((m0 x + m1 y) + m2 z) + m3 in float32 (numpy does not fuse)."""
    M = M.astype(np.float32)
    out = p.copy()
    for r in range(3):
        out[:, r] = ((M[r, 0] * p[:, 0] + M[r, 1] * p[:, 1]) + M[r, 2] * p[:, 2]) + M[r, 3]
    return out


def rotate_f32(M, n):
    M = M.astype(np.float32)
    out = n.copy()
    for r in range(3):
        out[:, r] = (M[r, 0] * n[:, 0] + M[r, 1] * n[:, 1]) + M[r, 2] * n[:, 2]
    return out


def surface(n, seed, noise=0.0):
    """Points of a bumpy height field z = f(x, y) (no rigid motion slides it onto itself) with their analytic normals,
    n x 4 float32 each."""
    rng = np.random.default_rng(seed)
    x, y = rng.uniform(-60, 60, n), rng.uniform(-60, 60, n)
    z = 10 * np.sin(x / 15) * np.cos(y / 20) + 0.004 * x * y + 50.0
    fx = (10 / 15) * np.cos(x / 15) * np.cos(y / 20) + 0.004 * y
    fy = -(10 / 20) * np.sin(x / 15) * np.sin(y / 20) + 0.004 * x
    P = np.zeros((n, 4), dtype=np.float32)
    P[:, 0], P[:, 1], P[:, 2] = x, y, z
    if noise:
        P[:, :3] += noise * rng.normal(size=(n, 3))
    d = np.stack([-fx, -fy, np.ones(n)], axis=1)
    N = np.zeros((n, 4), dtype=np.float32)
    N[:, :3] = d / np.linalg.norm(d, axis=1, keepdims=True)
    return P, N


def motion(rotvec, t):
    M = np.eye(4)
    M[:3, :3] = Rotation.from_rotvec(rotvec).as_matrix()
    M[:3, 3] = t
    return M


# ---- CPU ----------------------------------------------------------------------------------------------------------------
def test_oracle_step_matches_numpy(sym):
    rng = np.random.default_rng(7)
    k = 400
    src = np.zeros((k, 4), np.float32); tgt = np.zeros((k, 4), np.float32)
    src[:, :3] = rng.uniform(-50, 50, (k, 3)); tgt[:, :3] = src[:, :3] + rng.normal(0, 0.5, (k, 3))
    n1 = np.zeros((k, 4), np.float32); n2 = np.zeros((k, 4), np.float32)
    a = rng.normal(size=(k, 3)); a /= np.linalg.norm(a, axis=1, keepdims=True)
    b = a + rng.normal(0, 0.1, (k, 3)); b /= np.linalg.norm(b, axis=1, keepdims=True)
    n1[:, :3] = a; n2[:, :3] = b
    n2[::3, :3] *= -1            # opposite directions: n = n1 - n2
    n1[5, 1] = np.nan            # skipped pair
    n2[11, 2] = np.inf           # skipped pair
    q = np.arange(k, dtype=np.int32)[::-1].copy()
    m = np.arange(k, dtype=np.int32)[::-1].copy()
    rc, T, x = sym.estimate_symmetric(src, n1, tgt, n2, q, m)
    assert rc == 0
    f = lambda a: a[q, :3].astype(np.float64)
    Tn, xn = np_symmetric_step(f(src), f(n1), tgt[m, :3].astype(np.float64), n2[m, :3].astype(np.float64))
    assert np.allclose(x, xn, rtol=1e-9, atol=1e-12)
    assert np.allclose(T, Tn, rtol=1e-9, atol=1e-11)
    # enforce_same_direction_normals: the step does not depend on which way the target normals face
    n2f = n2.copy(); n2f[::3, :3] *= -1
    _, T2, _ = sym.estimate_symmetric(src, n1, tgt, n2f, q, m)
    assert np.array_equal(T2, T)
    # degenerate: every normal equal and every pair on one plane -> not SPD
    flat = np.zeros((k, 4), np.float32); flat[:, 2] = 1.0
    pl = src.copy(); pl[:, 2] = 0.0
    rc, _, _ = sym.estimate_symmetric(pl, flat, pl, flat, q, m)
    assert rc == 1


def test_symmetric_pose_construction_matches_scipy(sym):
    rng = np.random.default_rng(3)
    k = 300
    src = np.zeros((k, 4), np.float32); src[:, :3] = rng.uniform(-20, 20, (k, 3))
    M = motion([0.05, -0.03, 0.02], [0.4, -0.2, 0.3])
    tgt = src.copy(); tgt[:, :3] = (src[:, :3].astype(np.float64) @ M[:3, :3].T + M[:3, 3]).astype(np.float32)
    nrm = np.zeros((k, 4), np.float32)
    d = rng.normal(size=(k, 3)); nrm[:, :3] = d / np.linalg.norm(d, axis=1, keepdims=True)
    tn = nrm.copy(); tn[:, :3] = nrm[:, :3] @ M[:3, :3].T
    idx = np.arange(k, dtype=np.int32)
    rc, T, x = sym.estimate_symmetric(src, nrm, tgt, tn, idx, idx)
    assert rc == 0
    R = Rotation.from_euler("ZYX", [x[2], x[1], x[0]])
    want = np.eye(4)
    want[:3, :3] = (R * R).as_matrix()
    want[:3, 3] = R.apply(x[3:])
    assert np.allclose(T, want, rtol=0, atol=1e-14)
    assert abs(np.linalg.det(T[:3, :3]) - 1) < 1e-12


def _np_icp_symmetric(src, sn, tgt, tn, guess, iters, max_dist, reciprocal):
    """numpy restatement of the oracle's loop: float32 points and normals moved in place by the float increment."""
    cur = xform_f32(guess, src)
    curn = rotate_f32(guess, sn)
    tt = cKDTree(tgt[:, :3].astype(np.float64))
    out = []
    for _ in range(iters):
        d, j = tt.query(cur[:, :3].astype(np.float64))
        keep = d * d <= max_dist * max_dist
        if reciprocal:
            st = cKDTree(cur[:, :3].astype(np.float64))
            _, back = st.query(tgt[j, :3].astype(np.float64))
            keep &= back == np.arange(len(cur))
        qi = np.nonzero(keep)[0]
        T, _ = np_symmetric_step(cur[qi, :3].astype(np.float64), curn[qi, :3].astype(np.float64),
                                 tgt[j[qi], :3].astype(np.float64), tn[j[qi], :3].astype(np.float64))
        Tf = T.astype(np.float32); Tf[3] = [0, 0, 0, 1]
        cur = xform_f32(Tf, cur)
        curn = rotate_f32(Tf, curn)
        out.append((len(qi), Tf.astype(np.float64)))
    return out


@pytest.mark.parametrize("reciprocal", [False, True])
def test_oracle_symmetric_loop_matches_numpy(orc, sym, reciprocal):
    src, sn = surface(1500, 1, noise=0.3)
    tgt0, tn0 = surface(1600, 2, noise=0.3)
    M = motion([0.01, -0.02, 0.015], [1.0, -2.0, 0.5])
    tgt = tgt0.copy(); tgt[:, :3] = (tgt0[:, :3].astype(np.float64) @ M[:3, :3].T + M[:3, 3]).astype(np.float32)
    tn = tn0.copy(); tn[:, :3] = (tn0[:, :3].astype(np.float64) @ M[:3, :3].T).astype(np.float32)
    tn[1::2, :3] *= -1   # half of the target normals face the other way
    guess = motion([0.002, 0.0, -0.001], [0.2, 0.1, 0.0]).astype(np.float32)
    iters, gate = 8, 6.0
    p = orc.make_params(max_iterations=iters, max_dist=gate, reciprocal=reciprocal, fixed_iterations=True, estimator=2)
    o = sym.icp_align(src, sn, tgt, tn, p, guess=guess)
    assert o["status"] == 0 and o["iterations"] == iters
    ref = _np_icp_symmetric(src, sn, tgt, tn, guess, iters, gate, reciprocal)
    for rec, (nc, Tf) in zip(o["log"], ref):
        assert rec["n_corr"] == nc
        assert np.allclose(rec["delta"], Tf, rtol=0, atol=2e-6)
    assert len(o["log"]) == iters


def test_noise_free_pair_recovers_the_motion(orc, sym):
    src, sn = surface(4000, 5)
    M = motion([0.01, -0.02, 0.015], [1.0, -2.0, 0.5])
    tgt = src.copy(); tgt[:, :3] = (src[:, :3].astype(np.float64) @ M[:3, :3].T + M[:3, 3]).astype(np.float32)
    tn = sn.copy(); tn[:, :3] = (sn[:, :3].astype(np.float64) @ M[:3, :3].T).astype(np.float32)
    p = orc.make_params(max_iterations=30, reciprocal=True, fixed_iterations=True, estimator=2)
    o = sym.icp_align(src, sn, tgt, tn, p)
    assert o["status"] == 0
    assert rot_angle(o["final"], M) <= 1e-6
    assert np.linalg.norm(o["final"][:3, 3] - M[:3, 3]) <= 1e-4
    assert o["n_corr"] == len(src)


def test_symmetric_exports(mvr, sym):
    assert mvr.SYMMETRIC == 2 and mvr.POINT_TO_PLANE == 1 and mvr.POINT_TO_POINT == 0
    L = mvr.lib()
    for name in ("mvr_set_source_normals", "mvr_normals_share"):
        assert hasattr(L, name), name
    assert hasattr(mvr.Context, "set_source_normals") and hasattr(mvr.Context, "normals_share")
    assert hasattr(sym.lib, "sym_estimate") and hasattr(sym.lib, "sym_icp_align")
    import os
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "mvr_b200.h")).read()
    assert "MVR_SYMMETRIC = 2" in hdr


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _pair(synth, V, n, p=0):
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    t, s = p, (p + 1) % V
    return views[s], views[t], driver_guess(init[t], init[s])


def _sym_params(mvr, iters, reciprocal, fixed=True):
    return mvr.default_params(max_iterations=iters, max_dist=4.0, reciprocal=int(reciprocal), fixed_iterations=int(fixed),
                              estimator=mvr.SYMMETRIC)


def _check_against_oracle(ctx_res, log, o):
    assert ctx_res["status"] == 0 and o["status"] == 0
    assert len(log) == len(o["log"])
    for g, w in zip(log, o["log"]):
        assert g["n_corr"] == w["n_corr"], "iteration %d" % g["iteration"]
    assert rot_angle(ctx_res["final"], o["final"]) < ROT_TOL
    dt = np.linalg.norm(ctx_res["final"][:3, 3].astype(np.float64) - o["final"][:3, 3])
    assert dt <= TRANS_REL_TOL * max(1.0, float(np.linalg.norm(o["final"][:3, 3]))), dt


@pytest.mark.gpu
@pytest.mark.parametrize("n,iters,V", [(50_000, 10, 24), (200_000, 30, 24)])
@pytest.mark.parametrize("reciprocal", [True, False])
def test_single_align_matches_oracle_with_the_gpu_normals(mvr, orc, sym, synth, n, iters, V, reciprocal):
    src, tgt, guess = _pair(synth, V, n)
    c = mvr.Context(0)
    c.set_target(tgt); c.set_source(src)
    tn = c.estimate_normals(mvr.TARGET, len(tgt), 16)
    sn = c.estimate_normals(mvr.SOURCE, len(src), 16)
    p = _sym_params(mvr, iters, reciprocal)
    r = c.icp_align(p, guess=guess, n_source=len(src))
    log = c.iterations()
    op = orc.make_params(max_iterations=iters, max_dist=4.0, reciprocal=reciprocal, fixed_iterations=True, estimator=2)
    o = sym.icp_align(src, sn, tgt, tn, op, guess=guess, max_log=iters)
    _check_against_oracle(r, log, o)
    # a repeat is a fresh align from its guess: the source normals are gathered again from the view's own
    r2 = c.icp_align(p, guess=guess, n_source=len(src))
    assert np.array_equal(r2["final"], r["final"]) and r2["n_corr"] == r["n_corr"]
    c.close()


@pytest.mark.gpu
def test_source_normals_by_copy_estimate_or_share_give_the_same_bits(mvr, synth):
    src, tgt, guess = _pair(synth, 24, 30_000)
    p = _sym_params(mvr, 8, True)
    a = mvr.Context(0)
    a.set_target(tgt); a.set_source(src)
    tn = a.estimate_normals(mvr.TARGET, len(tgt), 16)
    sn = a.estimate_normals(mvr.SOURCE, len(src), 16)
    ra = a.icp_align(p, guess=guess, n_source=len(src))
    b = mvr.Context(0)
    b.set_target(tgt); b.set_source(src)
    b.set_target_normals(tn); b.set_source_normals(sn)
    rb = b.icp_align(p, guess=guess, n_source=len(src))
    # the source view is the target of another context: its normals are shared, not estimated again
    d = mvr.Context(0)
    d.set_target(src)
    assert np.array_equal(d.estimate_normals(mvr.TARGET, len(src), 16).view(np.uint32), sn.view(np.uint32))
    c = mvr.Context(0)
    c.set_target(tgt); c.set_source(src)
    c.normals_share(mvr.TARGET, a, mvr.TARGET)
    c.normals_share(mvr.SOURCE, d, mvr.TARGET)
    rc = c.icp_align(p, guess=guess, n_source=len(src))
    for r in (rb, rc):
        assert r["status"] == 0
        assert np.array_equal(r["final"].view(np.uint32), ra["final"].view(np.uint32)) and r["n_corr"] == ra["n_corr"] and r["mse"] == ra["mse"]
    # the shared normals stay as they were: the align turned a copy
    assert np.array_equal(d.estimate_normals(mvr.TARGET, len(src), 16).view(np.uint32), sn.view(np.uint32))
    for x in (a, b, c, d):
        x.close()


@pytest.mark.gpu
def test_missing_normals_are_no_input(mvr, synth):
    src, tgt, guess = _pair(synth, 24, 20_000)
    p = _sym_params(mvr, 4, True)
    c = mvr.Context(0)
    c.set_target(tgt); c.set_source(src)

    def align_status():
        with pytest.raises(mvr.MvrError) as e:
            c.icp_align(p, guess=guess, n_source=len(src))
        return e.value.status, c.last_error()

    st, msg = align_status()
    assert st == mvr.ERR_NO_INPUT and "target normals" in msg
    c.estimate_normals(mvr.TARGET, len(tgt), 16)
    st, msg = align_status()
    assert st == mvr.ERR_NO_INPUT and "source normals" in msg
    sn = c.estimate_normals(mvr.SOURCE, len(src), 16)
    assert c.icp_align(p, guess=guess, n_source=len(src))["status"] == 0
    c.set_source(src)                      # a new source drops its normals
    st, msg = align_status()
    assert st == mvr.ERR_NO_INPUT and "source normals" in msg
    c.set_source_normals(sn)
    c.set_target(tgt)                      # a new target drops its normals
    st, msg = align_status()
    assert st == mvr.ERR_NO_INPUT and "target normals" in msg
    # only source normals: point-to-plane still needs target normals
    with pytest.raises(mvr.MvrError) as e:
        c.icp_align(mvr.default_params(max_iterations=2, max_dist=4.0, estimator=mvr.POINT_TO_PLANE), guess=guess, n_source=len(src))
    assert e.value.status == mvr.ERR_NO_INPUT
    # sharing: from a context without such normals, and between clouds of different sizes
    other = mvr.Context(0)
    other.set_target(src[:-5])
    with pytest.raises(mvr.MvrError) as e:
        c.normals_share(mvr.TARGET, other, mvr.TARGET)
    assert e.value.status == mvr.ERR_NO_INPUT
    with pytest.raises(mvr.MvrError) as e:
        c.normals_share(mvr.SOURCE, other, mvr.SOURCE)
    assert e.value.status == mvr.ERR_NO_INPUT
    other.estimate_normals(mvr.TARGET, len(src) - 5, 16)
    with pytest.raises(mvr.MvrError) as e:
        c.normals_share(mvr.SOURCE, other, mvr.TARGET)
    assert e.value.status == mvr.ERR_BAD_ARG
    with pytest.raises(mvr.MvrError) as e:
        c.set_source_normals(sn[:-1])
    assert e.value.status == mvr.ERR_BAD_ARG
    # a same-sized cloud's normals are shared
    third = mvr.Context(0)
    third.set_target(src)
    third.estimate_normals(mvr.TARGET, len(src), 16)
    c.set_source(src)
    c.normals_share(mvr.SOURCE, third, mvr.TARGET)
    c.estimate_normals(mvr.TARGET, len(tgt), 16)
    assert c.icp_align(p, guess=guess, n_source=len(src))["status"] == 0
    for x in (other, third, c):
        x.close()


@pytest.mark.gpu
def test_batch_equals_single_aligns_and_any_grouping(mvr, synth):
    V, n = 6, 20_000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    P = 5
    ctxs = [mvr.Context(0) for _ in range(P)]
    guesses = []
    for k, c in enumerate(ctxs):
        c.set_target(views[k]); c.set_source(views[k + 1])
        c.estimate_normals(mvr.TARGET, n, 16); c.estimate_normals(mvr.SOURCE, n, 16)
        guesses.append(driver_guess(init[k], init[k + 1]))
    p = _sym_params(mvr, 12, True)
    one = [c.icp_align(p, guess=g, n_source=n) for c, g in zip(ctxs, guesses)]
    for group in (0, 1, 2, 5):
        ctxs[0].set_batch_group(group)
        got = mvr.icp_align_batch(ctxs, p, guesses=guesses)
        for a, b in zip(got, one):
            assert a["status"] == 0
            assert np.array_equal(a["final"], b["final"]) and a["n_corr"] == b["n_corr"] and a["mse"] == b["mse"], group
    # with the convergence criteria on, too
    pc = _sym_params(mvr, 50, True, fixed=False)
    pc.transformation_epsilon = 1e-8
    one = [c.icp_align(pc, guess=g, n_source=n) for c, g in zip(ctxs, guesses)]
    ctxs[0].set_batch_group(2)
    got = mvr.icp_align_batch(ctxs, pc, guesses=guesses)
    for a, b in zip(got, one):
        assert np.array_equal(a["final"], b["final"]) and a["iterations"] == b["iterations"]
    for c in ctxs:
        c.close()


def _sym_tp(mvr, synth, **kw):
    icp = mvr.default_params(max_iterations=10, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=mvr.SYMMETRIC)
    return mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=2, mode=mvr.RING_PAIRS, loop_closure=1, **kw)


@pytest.fixture(scope="module")
def seq(synth):
    V, n = 6, 8000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    return V, n, views, poses, init


@pytest.mark.gpu
def test_ring_symmetric_equals_hand_built_pairs_and_is_invariant(mvr, synth, seq):
    V, n, views, poses, init = seq
    tp = _sym_tp(mvr, synth)
    reg1 = mvr.Registrator(0, 1)
    abs1, rep1 = reg1.register_turntable(views, tp, init_poses=init)
    c = mvr.Context(0)
    for p in range(V):
        t, s = p, (p + 1) % V
        assert rep1[p]["status"] == 0 and rep1[p]["iterations"] == 20
        c.set_target(views[t]); c.set_source(views[s])
        c.estimate_normals(mvr.TARGET, n, 16); c.estimate_normals(mvr.SOURCE, n, 16)
        r = c.icp_align(tp.icp, guess=driver_guess(init[t], init[s]), n_source=n)
        r = c.icp_align(tp.icp, guess=r["final"], n_source=n)
        assert np.array_equal(rep1[p]["pose"], r["final"]) and rep1[p]["n_corr"] == r["n_corr"] and rep1[p]["mse"] == r["mse"], "pair %d" % p
    c.close()
    # symmetric is its own estimator: other poses than point-to-plane
    icp_l = mvr.default_params(max_iterations=10, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=mvr.POINT_TO_PLANE)
    tpl = mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp_l, repeat_times=2, mode=mvr.RING_PAIRS, loop_closure=1)
    _, repl = reg1.register_turntable(views, tpl, init_poses=init)
    assert any(not np.array_equal(a["pose"], b["pose"]) for a, b in zip(repl, rep1))
    # streams, grouping and pair-range shards: bit-identical pair and absolute poses
    reg3 = mvr.Registrator(0, 3)
    abs3, rep3 = reg3.register_turntable(views, tp, init_poses=init)
    regg = mvr.Registrator(0, 1)
    regg.context(0).set_batch_group(1)
    absg, repg = regg.register_turntable(views, tp, init_poses=init)
    for reps, abss in ((rep3, abs3), (repg, absg)):
        for p in range(V):
            assert np.array_equal(rep1[p]["pose"], reps[p]["pose"]) and rep1[p]["n_corr"] == reps[p]["n_corr"]
        for v in range(V):
            assert np.array_equal(abs1[v], abss[v])
    # shards: (0, 2) ends at view 2, (2, 5) at view 5, (5, 6) at view 0 -- none of them has its last source as a target
    got = {}
    for lo, hi in ((0, 2), (2, 5), (5, 6)):
        need = {q % V for p in range(lo, hi) for q in (p, p + 1)}
        _, reps = reg3.register_turntable([views[v] if v in need else None for v in range(V)], _sym_tp(mvr, synth, pair_begin=lo, pair_end=hi),
                                          init_poses=init)
        for p in range(lo, hi):
            got[p] = reps[p]
    for p in range(V):
        assert np.array_equal(got[p]["pose"], rep1[p]["pose"]) and got[p]["status"] == 0 and got[p]["n_corr"] == rep1[p]["n_corr"]
    # an empty view: its pairs report MVR_ERR_NO_INPUT and keep their guesses, the others align
    holed = list(views); holed[3] = np.zeros((0, 4), dtype=np.float32)
    _, reph = reg1.register_turntable(holed, tp, init_poses=init)
    assert [r["status"] for r in reph] == [0, 0, mvr.ERR_NO_INPUT, mvr.ERR_NO_INPUT, 0, 0]
    for p in (0, 1, 4, 5):
        assert np.array_equal(reph[p]["pose"], rep1[p]["pose"])
    for r in (reg1, reg3, regg):
        r.close()


@pytest.mark.gpu
def test_multi_gpu_symmetric_matches_the_single_gpu_ring(mvr, synth):
    import torch
    import mvr_b200.ring as ring
    V, n = 8, 20_000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    icp = mvr.default_params(max_iterations=10, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=mvr.SYMMETRIC)
    tp = mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1)
    reg = mvr.Registrator(0, 1)
    one_poses, one_reps = reg.register_turntable(views, tp, init_poses=init)
    reg.close()
    assert all(r["status"] == 0 for r in one_reps)
    want = ring.pose_checksum(ring.pack_reports(one_reps, 0, V))
    for g in [1] + [g for g in (2, 4, 8) if g <= torch.cuda.device_count()]:
        m = mvr.MultiRegistrator(range(g))
        got_poses, reps, recs, _ = m.register_turntable(views, tp, init_poses=init)
        assert ring.pose_checksum(recs) == want, "%d GPUs: pair records differ from the single-GPU run" % g
        for a, b in zip(reps, one_reps):
            assert np.array_equal(a["pose"], b["pose"]) and a["n_corr"] == b["n_corr"] and a["mse"] == b["mse"]
        for a, b in zip(got_poses, one_poses):
            assert np.array_equal(a, b)
        m.close()


@pytest.mark.gpu
def test_bench_size_symmetric_ring_is_at_least_as_accurate_as_point_to_point(mvr, synth):
    """24 views x 200k points, reciprocal, max_dist 4, 30 fixed iterations: every pair aligns, and the median pair rotation
    error against the synthetic truth is no worse than point-to-point's on the same views."""
    V, n = 24, 200_000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    reg = mvr.Registrator(0, 1)
    med = {}
    for est in (mvr.POINT_TO_POINT, mvr.SYMMETRIC):
        icp = mvr.default_params(max_iterations=30, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=est)
        tp = mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1)
        _, rep = reg.register_turntable(views, tp, init_poses=init)
        assert all(r["status"] == 0 and r["iterations"] == 30 for r in rep)
        err = [rot_angle(rep[p]["pose"], np.linalg.inv(poses[p]) @ poses[(p + 1) % V]) for p in range(V)]
        med[est] = float(np.median(err))
    reg.close()
    assert med[mvr.SYMMETRIC] <= med[mvr.POINT_TO_POINT], med
