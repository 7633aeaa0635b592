"""Point-to-plane ring registration: the target normals of every ring pair come from one batched GPU pass
(mvr_estimate_normals_batch) and equal, bit for bit, what mvr_estimate_normals computes per cloud; the ring driver
(mvr_register_turntable, MVR_REGISTER_RING_PAIRS with icp.estimator = MVR_POINT_TO_PLANE) then gives each pair the
pose of a hand-built point-to-plane pair, whatever the streams, grouping, shards or GPU count."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ROT_TOL = 1e-5       # rad (north star)
TRANS_REL_TOL = 1e-6


def rot_angle(A, B):
    R = np.asarray(A, dtype=np.float64)[:3, :3] @ np.asarray(B, dtype=np.float64)[:3, :3].T
    w = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    return float(np.arcsin(min(1.0, np.linalg.norm(w))))


def driver_guess(init_t, init_s):
    """The ring driver's initial guess of a pair, in its arithmetic: float(inverseRigid(pose_t) * pose_s) in double, the sums
    in registrator.cpp's order."""
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


# ---- CPU: the ABI ------------------------------------------------------------------------------------------------------
def test_turntable_params_layout_matches_the_header(mvr, tmp_path):
    """mvr_turntable_params grew `normal_k` as its last field: the C compiler and the ctypes mirror agree on its size and offset."""
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "mvr_b200.h"\n'
                   'int main(void) { printf("%zu %zu\\n", sizeof(mvr_turntable_params), offsetof(mvr_turntable_params, normal_k)); return 0; }\n')
    exe = str(tmp_path / "layout")
    r = subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    size, off = (int(x) for x in subprocess.run([exe], capture_output=True, text=True, check=True).stdout.split())
    assert size == ctypes.sizeof(mvr.TurntableParams)
    assert off == mvr.TurntableParams.normal_k.offset
    assert mvr.TurntableParams._fields_[-1][0] == "normal_k"


def test_turntable_params_default_normal_k(mvr):
    assert mvr.turntable_params().normal_k == 16
    assert hasattr(mvr.lib(), "mvr_estimate_normals_batch")


# ---- GPU ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def seq(synth):
    V, n = 6, 8000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    return V, n, views, poses, init


def _targets(synth):
    """Targets of the batch test: two scans, a 3-point cloud, an empty one, a scan with non-finite points."""
    a, _ = synth.turntable_view(0, 24, 20_000)
    b, _ = synth.turntable_view(3, 24, 50_000)
    c = a[:3].copy()
    e = np.zeros((0, 4), dtype=np.float32)
    d, _ = synth.turntable_view(5, 24, 30_000)
    d = d.copy()
    d[::97, 0] = np.nan
    d[5::211, 2] = np.inf
    return [a, b, c, e, d]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [8, 16, 32])
def test_batch_normals_equal_single_normals_bit_for_bit(mvr, synth, k):
    tg = _targets(synth)
    vps = np.array([[0, 0, 0], [10, -20, 5], [1, 2, 3], [0, 0, 0], [-50, 0, 900]], dtype=np.float32)
    batch = [mvr.Context(0) for _ in tg]
    for c, t in zip(batch, tg):
        c.set_target(t)
    got = mvr.estimate_normals_batch(batch, k, viewpoints=vps, want=True)
    one = mvr.Context(0)
    for i, t in enumerate(tg):
        one.set_target(t)
        want = one.estimate_normals(mvr.TARGET, len(t), k, viewpoint=tuple(float(x) for x in vps[i]))
        assert got[i].shape == want.shape
        assert np.array_equal(got[i].view(np.uint32), want.view(np.uint32)), "target %d, k %d" % (i, k)
    assert np.all(np.isnan(got[4][::97]))
    # the normals stay on the device as the target normals: a point-to-plane align reads them, the same bits either way
    src, Ts = synth.turntable_view(1, 24, 20_000)
    guess = (synth.perturbation() @ Ts).astype(np.float32)
    p = mvr.default_params(max_iterations=6, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=mvr.POINT_TO_PLANE)
    batch[0].set_source(src)
    r_batch = batch[0].icp_align(p, guess=guess, n_source=len(src))
    one.set_target(tg[0]); one.set_source(src)
    one.estimate_normals(mvr.TARGET, len(tg[0]), k, viewpoint=(0.0, 0.0, 0.0))
    r_one = one.icp_align(p, guess=guess, n_source=len(src))
    assert r_batch["status"] == 0 and r_batch["n_corr"] > 0
    assert np.array_equal(r_batch["final"], r_one["final"]) and r_batch["n_corr"] == r_one["n_corr"]
    # a context without a target: MVR_ERR_NO_INPUT in its status, the others still complete
    missing = mvr.Context(0)
    ctxs = [batch[0], missing, batch[1]]
    hs = (ctypes.c_void_p * 3)(*[c._h for c in ctxs])
    outs = [np.full((len(tg[0]), 4), 7, np.float32), None, np.full((len(tg[1]), 4), 7, np.float32)]
    fpp = ctypes.POINTER(ctypes.c_float)
    ptrs = (fpp * 3)(*[o.ctypes.data_as(fpp) if o is not None else fpp() for o in outs])
    st = np.full(3, -1, dtype=np.int32)
    rc = mvr.lib().mvr_estimate_normals_batch(hs, 3, k, None, ptrs, st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
    assert rc == mvr.OK and list(st) == [mvr.OK, mvr.ERR_NO_INPUT, mvr.OK]
    one.set_target(tg[1])
    assert np.array_equal(outs[2].view(np.uint32), one.estimate_normals(mvr.TARGET, len(tg[1]), k).view(np.uint32))
    with pytest.raises(mvr.MvrError) as e:
        mvr.estimate_normals_batch(ctxs, k)
    assert e.value.status == mvr.ERR_NO_INPUT
    # batch-level argument errors
    with pytest.raises(mvr.MvrError) as e:
        mvr.estimate_normals_batch([batch[0], batch[0]], k)
    assert e.value.status == mvr.ERR_BAD_ARG
    with pytest.raises(mvr.MvrError) as e:
        mvr.estimate_normals_batch(batch[:2], 2)
    assert e.value.status == mvr.ERR_BAD_ARG
    for c in batch + [one, missing]:
        c.close()


def _p2l_tp(mvr, synth, **kw):
    icp = mvr.default_params(max_iterations=10, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=mvr.POINT_TO_PLANE)
    return mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=2, mode=mvr.RING_PAIRS, loop_closure=1, **kw)


@pytest.mark.gpu
def test_ring_point_to_plane_equals_hand_built_pairs_and_is_invariant(mvr, synth, seq):
    V, n, views, poses, init = seq
    tp = _p2l_tp(mvr, synth)
    reg1 = mvr.Registrator(0, 1)
    abs1, rep1 = reg1.register_turntable(views, tp, init_poses=init)
    icp = tp.icp
    c = mvr.Context(0)
    for p in range(V):
        t, s = p, (p + 1) % V
        assert rep1[p]["status"] == 0 and rep1[p]["iterations"] == 20
        c.set_target(views[t]); c.set_source(views[s])
        c.estimate_normals(mvr.TARGET, n, 16, viewpoint=(0.0, 0.0, 0.0))
        r = c.icp_align(icp, guess=driver_guess(init[t], init[s]), n_source=n)
        r = c.icp_align(icp, guess=r["final"], n_source=n)
        assert np.array_equal(rep1[p]["pose"], r["final"]) and rep1[p]["n_corr"] == r["n_corr"] and rep1[p]["mse"] == r["mse"], "pair %d" % p
    c.close()
    # normal_k = 0 means 16; out of range is refused
    _, rep0 = reg1.register_turntable(views, _p2l_tp(mvr, synth, normal_k=0), init_poses=init)
    assert all(np.array_equal(a["pose"], b["pose"]) for a, b in zip(rep0, rep1))
    for bad in (2, 33, -1):
        with pytest.raises(mvr.MvrError) as e:
            reg1.register_turntable(views, _p2l_tp(mvr, synth, normal_k=bad), init_poses=init)
        assert e.value.status == mvr.ERR_BAD_ARG
    # another k gives other normals, hence other poses
    _, rep8 = reg1.register_turntable(views, _p2l_tp(mvr, synth, normal_k=8), init_poses=init)
    assert any(not np.array_equal(a["pose"], b["pose"]) for a, b in zip(rep8, rep1))
    # streams, grouping and pair-range shards: bit-identical pair and absolute poses
    reg3 = mvr.Registrator(0, 3)
    abs3, rep3 = reg3.register_turntable(views, tp, init_poses=init)
    for p in range(V):
        assert np.array_equal(rep1[p]["pose"], rep3[p]["pose"]) and rep1[p]["n_corr"] == rep3[p]["n_corr"]
    for v in range(V):
        assert np.array_equal(abs1[v], abs3[v])
    regg = mvr.Registrator(0, 1)
    regg.context(0).set_batch_group(1)
    absg, repg = regg.register_turntable(views, tp, init_poses=init)
    for p in range(V):
        assert np.array_equal(rep1[p]["pose"], repg[p]["pose"]) and rep1[p]["n_corr"] == repg[p]["n_corr"]
    for v in range(V):
        assert np.array_equal(abs1[v], absg[v])
    got = {}
    for lo, hi in ((0, 2), (2, 5), (5, 6)):
        need = {q % V for p in range(lo, hi) for q in (p, p + 1)}
        _, reps = reg3.register_turntable([views[v] if v in need else None for v in range(V)], _p2l_tp(mvr, synth, pair_begin=lo, pair_end=hi),
                                          init_poses=init)
        for p in range(lo, hi):
            got[p] = reps[p]
    for p in range(V):
        assert np.array_equal(got[p]["pose"], rep1[p]["pose"]) and got[p]["status"] == 0
    radius = 0.5 * float((views[0][:, :3].max(axis=0) - views[0][:, :3].min(axis=0)).max())
    closed = mvr.ring_close([got[p]["pose"] for p in range(V)], [got[p]["n_corr"] for p in range(V)], relax=True, iterations=16,
                            centre=synth.PIVOT, rot_scale=radius)
    for v in range(V):
        assert np.array_equal(closed[v], abs1[v])
    # an empty view keeps its meaning: its pairs report MVR_ERR_NO_INPUT and keep their guesses, the others align
    holed = list(views); holed[3] = np.zeros((0, 4), dtype=np.float32)
    _, reph = reg1.register_turntable(holed, tp, init_poses=init)
    assert [r["status"] for r in reph] == [0, 0, mvr.ERR_NO_INPUT, mvr.ERR_NO_INPUT, 0, 0]
    assert np.array_equal(reph[2]["pose"], driver_guess(init[2], init[3]))
    for p in (0, 1, 4, 5):
        assert np.array_equal(reph[p]["pose"], rep1[p]["pose"])
    for r in (reg1, reg3, regg):
        r.close()


@pytest.mark.gpu
def test_ring_point_to_plane_matches_oracle_with_the_gpu_normals(mvr, orc, synth, seq):
    """Each ring pair against the oracle's point-to-plane ICP given the GPU's own target normals (read back through the batch's
    host copies): the comparison is about ICP only."""
    V, n, views, poses, init = seq
    tp = _p2l_tp(mvr, synth)
    reg = mvr.Registrator(0, 1)
    _, rep = reg.register_turntable(views, tp, init_poses=init)
    reg.close()
    ctxs = [mvr.Context(0) for _ in range(V)]
    for c, v in zip(ctxs, views):
        c.set_target(v)
    nrm = mvr.estimate_normals_batch(ctxs, 16, want=True)
    op = orc.make_params(max_iterations=10, max_dist=4.0, reciprocal=True, fixed_iterations=True, estimator=1)
    for p in range(V):
        t, s = p, (p + 1) % V
        o = orc.icp_align(views[s], views[t], op, guess=driver_guess(init[t], init[s]), tgt_normals=nrm[t])
        o = orc.icp_align(views[s], views[t], op, guess=o["final"], tgt_normals=nrm[t])
        assert rep[p]["n_corr"] == o["n_corr"], "pair %d" % p
        assert rot_angle(rep[p]["pose"], o["final"]) < ROT_TOL
        dt = np.linalg.norm(rep[p]["pose"][:3, 3].astype(np.float64) - o["final"][:3, 3])
        assert dt <= TRANS_REL_TOL * max(1.0, float(np.linalg.norm(o["final"][:3, 3]))), (p, dt)
    for c in ctxs:
        c.close()


@pytest.mark.gpu
def test_multi_gpu_point_to_plane_matches_the_single_gpu_ring(mvr, synth):
    import torch
    import mvr_b200.ring as ring
    V, n = 8, 20_000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    icp = mvr.default_params(max_iterations=10, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=mvr.POINT_TO_PLANE)
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
def test_bench_size_point_to_plane_ring_is_at_least_as_accurate_as_point_to_point(mvr, synth):
    """24 views x 200k points, reciprocal, max_dist 4, 30 fixed iterations: every pair aligns, and the median pair rotation
    error against the synthetic truth is no worse than point-to-point's on the same views."""
    V, n = 24, 200_000
    views, poses = synth.turntable_sequence(V, n)
    E = synth.perturbation()
    init = [(poses[v] @ E) if v % 2 else poses[v].copy() for v in range(V)]
    reg = mvr.Registrator(0, 1)
    med = {}
    for est in (mvr.POINT_TO_POINT, mvr.POINT_TO_PLANE):
        icp = mvr.default_params(max_iterations=30, max_dist=4.0, reciprocal=1, fixed_iterations=1, estimator=est)
        tp = mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1)
        _, rep = reg.register_turntable(views, tp, init_poses=init)
        assert all(r["status"] == 0 and r["iterations"] == 30 for r in rep)
        err = [rot_angle(rep[p]["pose"], np.linalg.inv(poses[p]) @ poses[(p + 1) % V]) for p in range(V)]
        med[est] = float(np.median(err))
    reg.close()
    assert med[mvr.POINT_TO_PLANE] <= med[mvr.POINT_TO_POINT], med
