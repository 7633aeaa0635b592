"""Global registration without an initial guess (mvr_global_align) on the B200: stage times, success rate over seeded placements
and the scorer's speed on far-off hypotheses.

Workloads (synth.py, object ~200 mm across, 0.2 mm noise):
  view  -- two partial turntable views 45 degrees apart, 200k points each; the source is moved by a seeded arbitrary placement.
  ring  -- two merged 12-view rings of 200k-point views (2.4M points each): ring A in the table's placement, ring B in a seeded
           arbitrary placement, each registered with register_turntable (point-to-point ring) and posed with apply_pose.
Stages: the keypoint features of each cloud (Context.fpfh), the mutual match (Context.match_features), the whole global_align
(wall clock); its device spans (report gpu_ms: features + match + scoring, CUDA events) and the kernel statistics (normals =
features, nn = match + scoring) with profiling on in a separate call; host draws = wall - device spans; the point-to-plane
refine (target normals + mvr_icp_align from the returned pose).  Success: the returned pose within 5 degrees and 5 mm at the
object centre, and the refined pose within 2e-3 rad and 1 mm.

Usage: python scripts/bench_global.py [--placements 16] [--out-dir profiles]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mvr_b200 as mvr            # noqa: E402
import mvr_b200.synth as synth    # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:   # the numbers still stand, but without the card they are not comparable
        return dict(error=str(e))


def rot_angle(A, B):
    R = np.asarray(A, dtype=np.float64)[:3, :3] @ np.asarray(B, dtype=np.float64)[:3, :3].T
    return float(np.arccos(np.clip((np.trace(R) - 1.0) / 2.0, -1.0, 1.0)))


def centre_error(A, B, c):
    c = np.append(np.asarray(c, dtype=np.float64), 1.0)
    return float(np.linalg.norm((np.asarray(A, dtype=np.float64) @ c - np.asarray(B, dtype=np.float64) @ c)[:3]))


def place(pts, P):
    out = pts.copy()
    out[:, :3] = (pts[:, :3].astype(np.float64) @ P[:3, :3].T + P[:3, 3]).astype(np.float32)
    return out


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, 1e3 * (time.perf_counter() - t0)


def run_case(tgt, src, truth, centre, vp, prm, detail):
    c = mvr.Context(0)
    c.set_target(tgt); c.set_source(src)
    rec = {}
    if detail:
        c.fpfh(mvr.TARGET, prm.keypoints, prm.k)   # warm-up of every shape
        (_, _, ft), rec["features_target_ms"] = timed(lambda: c.fpfh(mvr.TARGET, prm.keypoints, prm.k))
        (_, _, fs), rec["features_source_ms"] = timed(lambda: c.fpfh(mvr.SOURCE, prm.keypoints, prm.k))
        _, rec["match_ms"] = timed(lambda: c.match_features(fs, ft))
        c.global_align(prm)
    (pose, rep), wall = timed(lambda: c.global_align(prm))
    rec.update(global_align_ms=wall, device_spans_ms=rep["gpu_ms"], host_draws_ms=wall - rep["gpu_ms"], report=rep)
    if detail:
        c.set_profiling(True)
        c.kernel_stats(reset=True)
        c.global_align(prm)
        st = c.kernel_stats(reset=True)
        c.set_profiling(False)
        rec["kernel_ms"] = {k: st[k]["ms"] for k in ("normals", "nn", "sort", "table")}
        rec["scoring_ms"] = st["nn"]["ms"]   # match + scoring kernels; the match alone is match_ms (with its copies)
    rec["rot_err_deg"] = float(np.degrees(rot_angle(pose, truth)))
    rec["centre_err_mm"] = centre_error(pose, truth, centre)
    _, rec["target_normals_ms"] = timed(lambda: c.estimate_normals(mvr.TARGET, len(tgt), 16, viewpoint=vp))
    p = mvr.default_params(max_iterations=60, max_dist=4.0, reciprocal=0, estimator=mvr.POINT_TO_PLANE, transformation_epsilon=1e-10)
    r, rec["refine_ms"] = timed(lambda: c.icp_align(p, guess=pose, n_source=len(src)))
    rec["refine_iterations"] = r["iterations"]
    rec["refined_rot_err_rad"] = rot_angle(r["final"], truth)
    rec["refined_centre_err_mm"] = centre_error(r["final"], truth, centre)
    rec["success"] = bool(rec["rot_err_deg"] < 5 and rec["centre_err_mm"] < 5 and rec["refined_rot_err_rad"] < 2e-3
                          and rec["refined_centre_err_mm"] < 1.0)
    c.close()
    return rec


def far_scoring(n=200_000, nc=1024, samples=4096):
    """k_score on hypotheses that put the samples far from the target surface, against near-correct ones (one call each)."""
    tgt, _ = synth.turntable_view(0, 8, n)
    src, T1 = synth.turntable_view(1, 8, n)
    near = np.stack([(synth.rotation_about_axis(np.deg2rad(d)) @ T1).astype(np.float32) for d in np.linspace(-3, 3, nc)])
    far = np.stack([(synth.random_placement(1000 + k) @ T1).astype(np.float32) for k in range(nc)])
    c = mvr.Context(0)
    c.set_target(tgt); c.set_source(src)
    out = {}
    for name, cands in (("near", near), ("far", far)):
        mvr.score_guesses_batch([c], cands[None], 4.0, samples)
        c.set_profiling(True)
        c.kernel_stats(reset=True)
        reps = 5
        for _ in range(reps):
            _, inl, _ = mvr.score_guesses_batch([c], cands[None], 4.0, samples)
        st = c.kernel_stats(reset=True)
        c.set_profiling(False)
        ms = st["nn"]["ms"] / reps
        q = float(st["nn"]["units"]) / reps
        out[name] = dict(kernel_ms=ms, queries=q, gqueries_per_s=q / ms / 1e6, inlier_fraction=float(inl.sum()) / (q or 1))
    c.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--placements", type=int, default=16)
    ap.add_argument("--out-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--skip-ring", action="store_true")
    a = ap.parse_args()
    os.makedirs(a.out_dir, exist_ok=True)
    info = gpu_info()
    prm = mvr.global_params()
    params = {f: getattr(prm, f) for f, _ in mvr.GlobalParams._fields_}
    res = dict(gpu=info, params=params)

    tgt, _ = synth.turntable_view(0, 8, 200_000)
    src0, T1 = synth.turntable_view(1, 8, 200_000)
    view = []
    for k in range(a.placements):
        P = synth.random_placement(100 + k)
        view.append(run_case(tgt, place(src0, P), T1 @ np.linalg.inv(P), P[:3, :3] @ synth.CENTER + P[:3, 3], np.zeros(3), prm, k == 0))
        print("view", k, json.dumps({x: view[-1][x] for x in ("global_align_ms", "rot_err_deg", "centre_err_mm", "success")}), flush=True)
    res["view"] = dict(points=200_000, cases=view, success=sum(r["success"] for r in view), of=len(view))

    if not a.skip_ring:
        V, n = 12, 200_000
        reg = mvr.Registrator(0)
        icp = mvr.default_params(max_iterations=30, max_dist=4.0, reciprocal=1, fixed_iterations=1)
        tp = mvr.turntable_params(pivot=synth.PIVOT, axis=synth.AXIS, icp=icp, repeat_times=1, mode=mvr.RING_PAIRS, loop_closure=1)
        ctx = mvr.Context(0)

        def merged_ring(placement):
            views, _ = synth.turntable_sequence(V, n, placement=placement)
            poses, _ = reg.register_turntable(views, tp)
            return np.concatenate([ctx.apply_pose(v, T.astype(np.float64)) for v, T in zip(views, poses)])

        ring_a = merged_ring(None)
        ring = []
        for k in range(a.placements):
            P = synth.random_placement(200 + k)
            ring.append(run_case(ring_a, merged_ring(P), np.linalg.inv(P), P[:3, :3] @ synth.CENTER + P[:3, 3], synth.CENTER, prm, k == 0))
            print("ring", k, json.dumps({x: ring[-1][x] for x in ("global_align_ms", "rot_err_deg", "centre_err_mm", "success")}), flush=True)
        res["ring"] = dict(points=len(ring_a), cases=ring, success=sum(r["success"] for r in ring), of=len(ring))
        ctx.close(); reg.close()

    res["scoring"] = far_scoring()
    print("scoring", json.dumps(res["scoring"]), flush=True)
    with open(os.path.join(a.out_dir, "global_bench.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(gpu=info, view_success=res["view"]["success"], ring_success=res.get("ring", {}).get("success"))))


if __name__ == "__main__":
    main()
